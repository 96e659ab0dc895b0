// cse_slots.cuh -- the level loop for HUGE frontiers (millions of nodes per round): warps that never wait.
// Included by cse.cu after its shared definitions (CseArgs, CseDeviceState, grid_barrier, cse_step, put_words).
//
// Why.  cse_wide_kernel fixes every output position with chained prefix sums inside the round, so a tile's flush waits
// for its CTA's slowest warp and for other CTAs' aggregates: measured (profiles/r2_cse_experiments.md) no unit of the SM
// or the memory system is busy and the round costs the same whatever is switched off -- each tile iteration lasts as
// long as the slowest of its ~100 memory requests.  A probe with fully independent warps ran the same round 1.55x faster.
//
// How.  A round is cut into chunks of SL_CH consecutive nodes of a level's ordered frontier; one warp takes a chunk from
// load to store and writes what it produces into SLOTS that belong to the chunk alone:
//     zero-children of chunk q of level l  ->  Z-slot q of level l+1   (SL_CH places, cz used)
//     one-children                          ->  O-slot q of level l+1
//     emitted words                         ->  E-slot of the chunk     (SL_CH * EW words, ce used)
// so nothing in phase A depends on another warp.  The next level's ordered frontier is then, by construction,
// Z-slot 0, Z-slot 1, ... , O-slot 0, O-slot 1, ... (bce.cpp:1275, 1283, 1339, 1346: zero-children list then one-children
// list, both in parent order) with holes; between two rounds the grid scans the slot counts (phase B):
//     P[c]      nodes before slot c            (so position g of the frontier is node g - P[c] of its slot c)
//     start[q]  the slot that holds position q * SL_CH   (where the next round's chunk q starts reading)
//     PE        words before a chunk's E-slot; the E-slots are copied to their final place in the stream buffer
// The frontier never moves: a round reads its nodes out of the slots through P / start (a handful of shuffles per
// chunk) and writes children once.  Three grid barriers per round instead of one -- nothing against rounds of a
// millisecond; smaller frontiers go back to the flat layout and cse_wide_kernel (cse_slots_to_flat / cse_flat_to_slots).
#pragma once

namespace bce {

#ifndef BCE_SL_ITEMS
#define BCE_SL_ITEMS 4
#endif
// nodes per lane x CTAs per SM, big rounds of the 1 GB input (ms): 4 x 4 (64 registers, 40 bytes spilled) 96.2 | 5 x 3: 98.9 |
// 3 x 4: 100.2 | 4 x 3 (78 registers): 101.0 | 5 x 4: 101.0 | 3 x 3: 109.1 | 2 x 4: 109.3 | 2 x 5: 109.6 | 6 x 2: 113.4
constexpr int SL_ITEMS = BCE_SL_ITEMS;
constexpr uint32_t SL_CH = 32 * SL_ITEMS;         // nodes per chunk = places per slot
#ifndef BCE_SL_MINB
#define BCE_SL_MINB 4
#endif
constexpr int SL_THREADS = 256, SL_WARPS = SL_THREADS / 32, SL_MINB = BCE_SL_MINB;

struct SlotLevel {               // one level's frontier in slot form
  uint32_t n;                    // nodes
  uint32_t nz;                   // ... of which in Z-slots (the zero-half); = P[sz], filled in by whoever loads the level
  uint32_t sz, so;               // number of Z-slots / O-slots; combined slot index c: [0, sz) Z, [sz, sz + so) O
  uint32_t zoff, ooff;           // first place of the Z / O slot regions in the node arena
  uint32_t doff;                 // first entry of the level's slot counts in cnt[] (P[] uses doff + level: one more per level)
  uint32_t soff;                 // first entry of the level's chunk starts in start[]
};
struct SlotState {               // lives in global memory, survives launches (drain / relaunch)
  SlotLevel lv[2][8];            // [round parity][level]
};
struct SlotArgs {
  uint32_t* ns[2]; uint32_t* na[2]; uint32_t* nb[2];   // node arenas (position, x0, x1) per round parity
  uint32_t arena_cap;            // places per arena
  uint8_t* cnt[2];               // slot fill counts per round parity
  uint32_t* P[2];                // exclusive scan of cnt per level (+1 entry per level)
  uint32_t* start[2];            // chunk -> slot of its first node
  uint32_t dir_cap;              // entries in cnt / P / start per parity
  uint32_t* eslot;               // E-slots of the current round: chunk t owns [t * SL_CH * EW, ...)
  uint16_t* ecnt;                // words in them
  uint32_t chunk_cap;            // chunks per round the E-slots / ecnt are sized for
  uint32_t* partial;             // [2][8][gridDim] phase-B partial sums (children, emitted words)
  SlotState* ss;
};

// One node per lane of a warp, the j-th of the chunk's lanes' nodes: its children go to the chunk's Z- and O-slot of
// the next level (places zbase / obase on, cz / co used so far) and its words to the chunk's E-slot (ce used), all in
// lane order, so the warp's nodes keep the order of the frontier.  EW = 5: raw counts, 5 words each; else one word, or
// three when k > 31.
template <int EW>
__device__ __forceinline__ void warp_slot_store(const CseStep& r, uint32_t x1, uint32_t x, unsigned lt_mask,
                                                uint32_t* __restrict__ gs, uint32_t* __restrict__ ga, uint32_t* __restrict__ gb,
                                                uint32_t zbase, uint32_t obase, uint32_t* __restrict__ ew,
                                                uint32_t& cz, uint32_t& co, uint32_t& ce) {
  const unsigned bz = __ballot_sync(0xffffffffu, r.z);
  const unsigned bo = __ballot_sync(0xffffffffu, r.o);
  const unsigned be = __ballot_sync(0xffffffffu, r.nw != 0u);
  if (r.z) { const uint32_t p = zbase + cz + __popc(bz & lt_mask); gs[p] = r.zs; ga[p] = r.za; gb[p] = r.zb; }
  if (r.o) { const uint32_t p = obase + co + __popc(bo & lt_mask); gs[p] = r.os; ga[p] = r.oa; gb[p] = r.ob; }
  cz += __popc(bz);
  co += __popc(bo);
  if (be) {
    if constexpr (EW == 5) {
      if (r.nw) put_words(ew + ce + 5u * __popc(be & lt_mask), r.nw, r.e0, r.e1, r.e2, x1, x);
      ce += 5u * __popc(be);
    } else {
      const unsigned b3 = __ballot_sync(0xffffffffu, r.nw == 3u);      // k > 31: two more words
      if (r.nw) put_words(ew + ce + __popc(be & lt_mask) + 2u * __popc(b3 & lt_mask), r.nw, r.e0, r.e1, r.e2, x1, x);
      ce += __popc(be) + 2u * __popc(b3);
    }
  }
}

__device__ __forceinline__ SlotLevel slot_level_load(const SlotLevel* p, const uint32_t* P, int level) {
  SlotLevel v;
  v.n = vol_load(&p->n);
  v.sz = vol_load(&p->sz); v.so = vol_load(&p->so);
  v.zoff = vol_load(&p->zoff); v.ooff = vol_load(&p->ooff);
  v.doff = vol_load(&p->doff); v.soff = vol_load(&p->soff);
  v.nz = P ? __ldcg(P + v.doff + level + v.sz) : vol_load(&p->nz);     // nodes before the first O-slot
  return v;
}

// ---- flat layout -> slots (host launches it before the first slot round) -----------------------------------------------
// Every level's zero-half becomes full Z-slots (the last one partly filled), its one-half -- stored back to front in the
// flat layout -- full O-slots.  P / start of this frontier are then produced by the kernel's phase B (first_scan).
__global__ void __launch_bounds__(256) cse_flat_to_slots_kernel(CseArgs a, SlotArgs sa) {
  __shared__ SlotLevel s_lv[8];
  CseDeviceState* S = a.st;
  const int par = S->round & 1;
  if (threadIdx.x == 0) {
    uint32_t place = 0, dir = 0, st = 0;
    for (int l = 0; l < 8; ++l) {
      SlotLevel v;
      const uint32_t cz = S->cnt[par][l][0], co = S->cnt[par][l][1];
      v.n = cz + co; v.nz = cz;
      v.sz = (cz + SL_CH - 1) / SL_CH; v.so = (co + SL_CH - 1) / SL_CH;
      v.zoff = place; place += v.sz * SL_CH;
      v.ooff = place; place += v.so * SL_CH;
      v.doff = dir; dir += v.sz + v.so;
      v.soff = st; st += v.sz + v.so + 1;
      s_lv[l] = v;
      if (blockIdx.x == 0) sa.ss->lv[par][l] = v;
    }
    if (place > sa.arena_cap || dir + 8 > sa.dir_cap || st > sa.dir_cap) atomicExch(&S->status, uint32_t(kCseOverflow));
  }
  __syncthreads();
  if (S->status == kCseOverflow) return;
  for (int l = 0; l < 8; ++l) {
    const SlotLevel v = s_lv[l];
    const uint32_t co = v.n - v.nz;
    for (uint32_t g = blockIdx.x * 256u + threadIdx.x; g < v.n; g += gridDim.x * 256u) {
      const bool one = g >= v.nz;
      const uint32_t from = flat_at(a.cap, v.nz, g);
      const uint32_t to = (one ? v.ooff : v.zoff) + (one ? g - v.nz : g);   // the g-th node of its half
      sa.ns[par][to] = a.fs[par][l][from];
      sa.na[par][to] = a.fa[par][l][from];
      sa.nb[par][to] = a.fb[par][l][from];
    }
    for (uint32_t c = blockIdx.x * 256u + threadIdx.x; c < v.sz + v.so; c += gridDim.x * 256u) {
      const bool one = c >= v.sz;
      const uint32_t k = one ? c - v.sz : c, half = one ? co : v.nz;
      sa.cnt[par][v.doff + c] = uint8_t(min(SL_CH, half - k * SL_CH));
    }
  }
}

// ---- slots -> flat layout (host launches it when the frontier has shrunk) ---------------------------------------------------
__global__ void __launch_bounds__(256) cse_slots_to_flat_kernel(CseArgs a, SlotArgs sa) {
  CseDeviceState* S = a.st;
  const int par = S->round & 1;
  const unsigned lane = threadIdx.x & 31;
  const uint32_t warps = gridDim.x * 8u, w0 = blockIdx.x * 8u + (threadIdx.x >> 5);
  for (int l = 0; l < 8; ++l) {
    const SlotLevel v = slot_level_load(&sa.ss->lv[par][l], sa.P[par], l);
    const uint32_t* __restrict__ P = sa.P[par] + v.doff + l;
    const uint32_t slots = v.sz + v.so;
    const uint32_t chunks = (v.n + 31u) / 32u;                         // 32 positions per warp step
    if (blockIdx.x == 0 && threadIdx.x == 0) { S->cnt[par][l][0] = v.nz; S->cnt[par][l][1] = v.n - v.nz; }
    for (uint32_t q = w0; q < chunks; q += warps) {
      const uint32_t g = q * 32u + lane;
      // binary search: last slot c with P[c] <= g (a frontier of this size is read once, no start table needed)
      uint32_t lo = 0, hi = slots;                                     // P has slots + 1 entries, P[slots] = n
      const uint32_t gg = min(g, v.n - 1u);
      while (hi - lo > 1u) {
        const uint32_t mid = (lo + hi) >> 1;
        if (P[mid] <= gg) lo = mid; else hi = mid;
      }
      if (g < v.n) {
        const uint32_t local = g - P[lo];
        const uint32_t from = v.zoff + lo * SL_CH + local;            // (the O-slots follow the Z-slots: ooff = zoff + sz * SL_CH)
        const uint32_t to = flat_at(a.cap, v.nz, g);
        a.fs[par][l][to] = sa.ns[par][from];
        a.fa[par][l][to] = sa.na[par][from];
        a.fb[par][l][to] = sa.nb[par][from];
      }
    }
  }
}

// ---- the round loop ----------------------------------------------------------------------------------------------------------
template <int EW>
__global__ void __launch_bounds__(SL_THREADS, SL_MINB) cse_slots_kernel(CseArgs a, SlotArgs sa, uint32_t first_scan) {
  __shared__ SlotLevel s_cur[8], s_nxt[8];
  __shared__ uint32_t s_tfirst[9];                  // first chunk of every level this round
  __shared__ uint32_t s_flags[2];
  __shared__ unsigned long long s_emitted[8];
  __shared__ uint32_t s_scan[SL_WARPS];
  __shared__ uint32_t s_base[8], s_ebase[8], s_total[8], s_etotal[8];
  __shared__ uint32_t s_pe[SL_THREADS];

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  CseDeviceState* S = a.st;
  SlotState* SS = sa.ss;
  const uint32_t G = gridDim.x;
  uint32_t round = vol_load(&S->round);
  const unsigned long long barrier0 = vol_load64(&S->barriers);
  uint32_t barriers_done = 0;                       // grid barriers passed by this launch
  if (vol_load(&S->status) == kCseOverflow) return;   // the conversion into slots did not fit: nobody touches the status
  if (blockIdx.x == 0 && tid == 0) S->status = kCseRunning;
  bool scan_only = first_scan != 0;                 // the frontier was just converted from the flat layout: build P / start first

  for (;;) {
    const int cur = round & 1, nxt = cur ^ 1;
    // ---- header: every CTA derives the same plan from the state in global memory --------------------------------
    if (tid < 8) {
      s_cur[tid] = slot_level_load(&SS->lv[cur][tid], scan_only ? nullptr : sa.P[cur], int(tid));
      s_emitted[tid] = vol_load64(&S->emitted[cur][tid]);
    }
    __syncthreads();
    if (tid == 0) {
      uint32_t t = 0, drain = 0, nch[8];
      unsigned long long nodes = 0;
      for (int l = 0; l < 8; ++l) {
        s_tfirst[l] = t;
        nch[l] = (s_cur[l].n + SL_CH - 1) / SL_CH;
        t += nch[l];
        nodes += s_cur[l].n;
        if (must_drain(s_emitted[l], s_cur[l].n, max_words(a), a.ecap[l], a.esoft[l])) drain = 1;
      }
      s_tfirst[8] = t;
      // where the children go: level L of the next round is fed by the chunks of level L - 1, one Z- and one O-slot each
      uint32_t place = 0, dir = 0, st = 0;
      for (int L = 0; L < 8; ++L) {
        SlotLevel v;
        v.n = v.nz = 0;
        v.sz = v.so = nch[(L + 7) & 7];
        v.zoff = place; place += v.sz * SL_CH;
        v.ooff = place; place += v.so * SL_CH;
        v.doff = dir; dir += v.sz + v.so;
        v.soff = st; st += v.sz + v.so + 1u;
        s_nxt[L] = v;
      }
      const bool overflow = place > sa.arena_cap || dir + 8u > sa.dir_cap || st > sa.dir_cap || t > sa.chunk_cap;
      s_flags[0] = t;
      // (leave: the host converts back to the flat layout)
      s_flags[1] = scan_only ? kCseRunning : round_status(nodes, round, a.round_limit, overflow, false, nodes < a.min_nodes, drain);
      if (blockIdx.x == 0 && s_flags[1] == kCseRunning && !scan_only) {
        S->visits += nodes;
        if (nodes > S->peak_frontier) S->peak_frontier = nodes;
      }
    }
    __syncthreads();
    const uint32_t total_chunks = s_flags[0];
    const uint32_t decision = s_flags[1];
    if (decision != kCseRunning) {
      if (blockIdx.x == 0 && tid == 0) { S->status = decision; S->round = round; S->barriers = barrier0 + barriers_done; }
      break;
    }
    const int pw = scan_only ? cur : nxt;             // the parity phase B works on
    if (!scan_only) {
      if (blockIdx.x == 0 && tid < 8) SS->lv[nxt][tid] = s_nxt[tid];   // n is filled in by phase B
      // ================= phase A: every warp on its own ============================================================
      // The chunk's place in the slots comes from two dependent loads (start[q], then the P window behind it) before
      // its nodes can even be asked for: both are fetched one / two chunks ahead, so that the chain a warp waits for is
      // nodes -> rank words only.
      const uint32_t stride = G * SL_WARPS;
      auto level_of = [&](uint32_t t) {                   // 3 compares: s_tfirst ascends
        int l = t >= s_tfirst[4] ? 4 : 0;
        l += t >= s_tfirst[l + 2] ? 2 : 0;
        l += t >= s_tfirst[l + 1] ? 1 : 0;
        return l;
      };
      auto load_start = [&](uint32_t t, int l) -> uint32_t {
        return t < total_chunks ? sa.start[cur][s_cur[l].soff + (t - s_tfirst[l])] : 0u;
      };
      auto load_window = [&](uint32_t t, int l, uint32_t base, uint32_t& p0, uint32_t& pw) {
        p0 = 0; pw = 0xFFFFFFFFu;
        if (t >= total_chunks) return;
        const uint32_t* __restrict__ P = sa.P[cur] + s_cur[l].doff + l;
        const uint32_t e = base + 1u + lane;
        p0 = P[base];
        if (e <= s_cur[l].sz + s_cur[l].so) pw = P[e];
      };
      uint32_t t = blockIdx.x * SL_WARPS + warp;
      int l = level_of(min(t, total_chunks - 1u)), l1 = level_of(min(t + stride, total_chunks - 1u));
      uint32_t cu_base = load_start(t, l), cu_p0, cu_pw;
      load_window(t, l, cu_base, cu_p0, cu_pw);
      uint32_t nx_base = load_start(t + stride, l1);
      for (; t < total_chunks; t += stride) {
        uint32_t n_p0, n_pw;
        load_window(t + stride, l1, nx_base, n_p0, n_pw);               // next chunk: its start arrived an iteration ago
        const int l2 = level_of(min(t + 2u * stride, total_chunks - 1u));
        const uint32_t nn_base = load_start(t + 2u * stride, l2);       // the one after: start only
        const int ln = (l + 1) & 7;
        const uint32_t q = t - s_tfirst[l];
        const SlotLevel v = s_cur[l];
        const uint32_t gbase = q * SL_CH, gend = min(v.n, gbase + SL_CH);          // frontier positions of the chunk
        const uint32_t slots = v.sz + v.so;
        const uint32_t* __restrict__ P = sa.P[cur] + v.doff + l;
        // --- where the chunk's nodes are: slot c and offset inside it for every position
        uint32_t c[SL_ITEMS], pc[SL_ITEMS], g[SL_ITEMS];
        uint32_t base = cu_base;
#pragma unroll
        for (int j = 0; j < SL_ITEMS; ++j) { g[j] = gbase + 32u * j + lane; c[j] = base; pc[j] = cu_p0; }
        uint32_t pwv = cu_pw;
        for (;;) {                                                      // windows of 32 following slots (one is the rule)
          const unsigned le = __ballot_sync(0xffffffffu, pwv < gend);   // slots that start inside the chunk
          const int nle = __popc(le);                                   // P ascends: they are the first nle lanes
          for (int i = 0; i < nle; ++i) {
            const uint32_t pv = __shfl_sync(0xffffffffu, pwv, i);
#pragma unroll
            for (int j = 0; j < SL_ITEMS; ++j)
              if (pv <= g[j]) { c[j] = base + 1u + i; pc[j] = pv; }
          }
          if (nle < 32) break;
          base += 32u;
          const uint32_t e = base + 1u + lane;
          pwv = e <= slots ? P[e] : 0xFFFFFFFFu;
        }
        cu_base = nx_base; cu_p0 = n_p0; cu_pw = n_pw; nx_base = nn_base;
        // --- nodes and their three rank words
        uint32_t ns[SL_ITEMS], na[SL_ITEMS], nb[SL_ITEMS];
        uint64_t wa[SL_ITEMS], wb[SL_ITEMS], wc[SL_ITEMS];
        const uint64_t* __restrict__ R = a.ranks[l];
#pragma unroll
        for (int j = 0; j < SL_ITEMS; ++j) {
          ns[j] = na[j] = nb[j] = 0;
          if (g[j] < gend) {
            const uint32_t at = v.zoff + c[j] * SL_CH + (g[j] - pc[j]);      // (the O-slots follow the Z-slots: ooff = zoff + sz * SL_CH)
            ns[j] = __ldcg(sa.ns[cur] + at);
            na[j] = __ldcg(sa.na[cur] + at);
            nb[j] = __ldcg(sa.nb[cur] + at);
          }
        }
#pragma unroll
        for (int j = 0; j < SL_ITEMS; ++j) {
          wa[j] = wb[j] = wc[j] = 0;
          if (g[j] < gend) rank_words(R, ns[j], na[j], nb[j], wa[j], wb[j], wc[j]);
        }
        // --- compute; outputs straight into the chunk's slots
        const SlotLevel nv = s_nxt[ln];
        uint32_t* __restrict__ gs = sa.ns[nxt];
        uint32_t* __restrict__ ga = sa.na[nxt];
        uint32_t* __restrict__ gb = sa.nb[nxt];
        const uint32_t zbase = nv.zoff + q * SL_CH, obase = nv.ooff + q * SL_CH;
        uint32_t* __restrict__ ew = sa.eslot + size_t(t) * (SL_CH * EW);
        const uint32_t one_base = a.C[ln];
        uint32_t cz = 0, co = 0, ce = 0;
#pragma unroll
        for (int j = 0; j < SL_ITEMS; ++j) {
          CseStep r{false, false, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          if (g[j] < gend) r = cse_step(a, l, one_base, ns[j], na[j], nb[j], wa[j], wb[j], wc[j]);
          warp_slot_store<EW>(r, nb[j], na[j] + nb[j], lt_mask, gs, ga, gb, zbase, obase, ew, cz, co, ce);
        }
        if (lane == 0) {
          sa.cnt[nxt][nv.doff + q] = uint8_t(cz);
          sa.cnt[nxt][nv.doff + nv.sz + q] = uint8_t(co);
          sa.ecnt[t] = uint16_t(ce);
        }
        l = l1; l1 = l2;
      }
      grid_barrier(S, barrier0 + barriers_done++, round);
    }

    // ================= phase B1: partial sums of this CTA's share of every level's slot counts =====================
    const SlotLevel* LV = scan_only ? s_cur : s_nxt;                  // levels being scanned (parity pw)
    uint32_t* const part_c = sa.partial;                              // [8][G] children
    uint32_t* const part_e = sa.partial + 8u * G;                     // [8][G] emitted words (level = emitting level)
    for (int L = 0; L < 8; ++L) {
      const uint32_t len = LV[L].sz + LV[L].so;
      const uint32_t per = (len + G - 1) / G;
      const uint32_t lo = min(len, blockIdx.x * per), hi = min(len, lo + per);
      const uint8_t* __restrict__ cn = sa.cnt[pw] + LV[L].doff;
      uint32_t sum = 0;
      for (uint32_t i = lo + tid; i < hi; i += SL_THREADS) sum += cn[i];
      uint32_t esum = 0;
      if (!scan_only) {                                               // E-slots of level L's chunks of THIS round
        const uint32_t elen = s_tfirst[L + 1] - s_tfirst[L];
        const uint32_t eper = (elen + G - 1) / G;
        const uint32_t elo = min(elen, blockIdx.x * eper), ehi = min(elen, elo + eper);
        for (uint32_t i = elo + tid; i < ehi; i += SL_THREADS) esum += sa.ecnt[s_tfirst[L] + i];
      }
      sum = __reduce_add_sync(0xffffffffu, sum);
      esum = __reduce_add_sync(0xffffffffu, esum);
      if (lane == 0) { s_scan[warp] = sum; s_pe[warp] = esum; }
      __syncthreads();
      if (tid == 0) {
        uint32_t a1 = 0, a2 = 0;
        for (int w = 0; w < SL_WARPS; ++w) { a1 += s_scan[w]; a2 += s_pe[w]; }
        part_c[L * G + blockIdx.x] = a1;
        part_e[L * G + blockIdx.x] = a2;
      }
      __syncthreads();
    }
    grid_barrier(S, barrier0 + barriers_done++, round);

    // ================= phase B2: bases, scans, chunk starts, emission to its final place ===========================
    for (int L = 0; L < 8; ++L) {                                     // this CTA's base = sum of the shares before it
      uint32_t b1 = 0, t1 = 0, b2 = 0, t2 = 0;
      for (uint32_t i = tid; i < G; i += SL_THREADS) {
        const uint32_t v1 = __ldcg(part_c + L * G + i), v2 = __ldcg(part_e + L * G + i);
        t1 += v1; t2 += v2;
        if (i < blockIdx.x) { b1 += v1; b2 += v2; }
      }
      b1 = __reduce_add_sync(0xffffffffu, b1); t1 = __reduce_add_sync(0xffffffffu, t1);
      b2 = __reduce_add_sync(0xffffffffu, b2); t2 = __reduce_add_sync(0xffffffffu, t2);
      __syncthreads();
      if (lane == 0) { s_scan[warp] = b1; s_pe[warp] = t1; s_pe[8 + warp] = b2; s_pe[16 + warp] = t2; }
      __syncthreads();
      if (tid == 0) {
        uint32_t x1 = 0, x2 = 0, x3 = 0, x4 = 0;
        for (int w = 0; w < SL_WARPS; ++w) { x1 += s_scan[w]; x2 += s_pe[w]; x3 += s_pe[8 + w]; x4 += s_pe[16 + w]; }
        s_base[L] = x1; s_total[L] = x2; s_ebase[L] = x3; s_etotal[L] = x4;
      }
      __syncthreads();
    }
    for (int L = 0; L < 8; ++L) {
      const SlotLevel v = LV[L];
      const uint32_t len = v.sz + v.so;
      const uint32_t per = (len + G - 1) / G;
      const uint32_t lo = min(len, blockIdx.x * per), hi = min(len, lo + per);
      const uint8_t* __restrict__ cn = sa.cnt[pw] + v.doff;
      uint32_t* __restrict__ Pw = sa.P[pw] + v.doff + L;
      uint32_t* __restrict__ stw = sa.start[pw] + v.soff;
      uint32_t run = s_base[L];
      for (uint32_t i0 = lo; i0 < hi; i0 += SL_THREADS) {
        const uint32_t i = i0 + tid;
        const uint32_t k = i < hi ? cn[i] : 0u;
        uint32_t tot;
        const uint32_t at = run + block_exclusive_scan<uint32_t, SL_THREADS>(k, s_scan, tot);
        if (i < hi) {
          Pw[i] = at;
          if (k) {                                                    // the slot holds positions [at, at + k): at most one chunk starts in it
            const uint32_t qn = (at + SL_CH - 1) / SL_CH;
            if (qn * SL_CH < at + k) stw[qn] = i;
          }
        }
        run += tot;
      }
      if (blockIdx.x == G - 1 && tid == 0) Pw[len] = s_total[L];
    }
    if (!scan_only) {
      for (int L = 0; L < 8; ++L) {                                   // level L's emitted words of this round
        const uint32_t elen = s_tfirst[L + 1] - s_tfirst[L];
        const uint32_t eper = (elen + G - 1) / G;
        const uint32_t elo = min(elen, blockIdx.x * eper), ehi = min(elen, elo + eper);
        const unsigned long long dst0 = s_emitted[L];
        uint32_t run = s_ebase[L];
        for (uint32_t i0 = elo; i0 < ehi; i0 += SL_THREADS) {
          const uint32_t i = i0 + tid;
          const uint32_t k = i < ehi ? sa.ecnt[s_tfirst[L] + i] : 0u;
          uint32_t tot;
          s_pe[tid] = run + block_exclusive_scan<uint32_t, SL_THREADS>(k, s_scan, tot);
          __syncthreads();
          const uint32_t nblk = min(uint32_t(SL_THREADS), ehi - i0);
          for (uint32_t j = warp; j < nblk; j += SL_WARPS) {          // one warp per chunk: its words are contiguous
            const uint32_t tch = s_tfirst[L] + i0 + j;
            const uint32_t kk = sa.ecnt[tch];
            const uint32_t* __restrict__ src = sa.eslot + size_t(tch) * (SL_CH * EW);
            uint32_t* __restrict__ dst = a.emit[L] + dst0 + s_pe[j];
            if (dst0 + s_pe[j] + kk <= a.ecap[L])
              for (uint32_t w = lane; w < kk; w += 32u) dst[w] = src[w];
          }
          __syncthreads();
          run += tot;
        }
      }
    }
    if (blockIdx.x == 0 && tid < 8) {
      const int L = tid;
      SS->lv[pw][L].n = s_total[L];
      S->cnt[pw][L][0] = s_total[L];                                   // the host only adds the two up; cse_slots_to_flat_kernel
      S->cnt[pw][L][1] = 0;                                            // writes the exact halves
      if (!scan_only) S->emitted[nxt][L] = s_emitted[L] + s_etotal[L];
    }
    grid_barrier(S, barrier0 + barriers_done++, round);
    if (scan_only) { scan_only = false; continue; }
    ++round;
    if (vol_load(&S->status) != kCseRunning || vol_load(&S->err) != 0) {
      if (blockIdx.x == 0 && tid == 0) { S->round = round; S->barriers = barrier0 + barriers_done; }
      break;
    }
  }
}

}  // namespace bce
