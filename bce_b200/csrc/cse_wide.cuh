// cse_wide.cuh -- the wide-frontier kernel of the CSE level loop, software pipelined.
// Included by cse.cu after its shared definitions (CseArgs, CseDeviceState, grid_barrier,
// load_items, cse_step, vol_load).
//
// Per round, per level, tiles of the ordered frontier; three prefix sums fix the positions of
// counts, zero- and one-children.  What matters is when things happen.  Measured on B200
// (profiles/): with every CTA resolving its
// chained scan right after computing a tile, the gridDim tiles in flight advance in lockstep
// (each waits for the aggregates of its same-phase predecessors) and the scan costs more than
// the rest of the round together.  So a tile's life is spread over two iterations:
//
//   iteration i    compute(i): flags, payloads, block scan; PUBLISH the tile aggregates;
//                  stage the compacted outputs in shared memory (buffer i & 1)
//                  load(i+1): node loads of this CTA's next tile
//                  resolve(i-1): chained scan for the PREVIOUS tile -- its predecessors
//                  published a whole iteration ago, so the walk does not wait
//                  gather(i+1): 3 rank-word gathers per node of the next tile
//                  flush(i-1): staged outputs of the previous tile to their final positions,
//                  contiguous runs instead of scattered 4-byte stores
//
// Tiles are handed out interleaved over the 8 levels (see locate), so that tiles running at
// the same time are links of 8 different chains rather than consecutive links of one.
#pragma once

namespace bce {

// EW = most words one count can take: 5 (raw bce_tuple) or 3 (packed modes); it sizes the staging
// buffers.  Both instances run 2 CTAs per SM: a 3-CTA build of the packed instance (80 registers)
// was measured 20 % slower on B200 (1 GB text: 206 ms against 175 ms for the level loop).
template <int ITEMS, int EW>
struct WideStage {                                  // one staging buffer
  static constexpr int TILE = CS_THREADS * ITEMS;
  uint32_t zs[TILE], za[TILE], zb[TILE];            // zero-children
  uint32_t os[TILE], oa[TILE], ob[TILE];            // one-children
  uint32_t e[TILE * EW];                            // emitted words
};

template <int ITEMS, int EW>
__global__ void __launch_bounds__(CS_THREADS, 512 / CS_THREADS) cse_wide_kernel(CseArgs a) {
  constexpr int TILE = CS_THREADS * ITEMS;
  extern __shared__ __align__(16) unsigned char wide_smem[];
  WideStage<ITEMS, EW>* stage = reinterpret_cast<WideStage<ITEMS, EW>*>(wide_smem);   // [2]
  __shared__ uint64_t s_scan[CS_THREADS / 32];
  __shared__ uint32_t s_prefix[3];
  __shared__ uint32_t s_cnt[8][2];
  __shared__ uint32_t s_tstart[8][2];
  __shared__ unsigned long long s_emitted[8];
  __shared__ uint32_t s_flags[2];
  __shared__ uint32_t s_lt[8], s_srt[8], s_cum[9];               // interleaved tile schedule (see locate)
  constexpr int SCHED_CAP = 1024;                                // this CTA's first tiles of a round, located once
  __shared__ uint32_t s_sched[SCHED_CAP];                        // (level << 28) | row in the level's chain

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  CseDeviceState* S = a.st;
  uint32_t round = vol_load(&S->round);
  uint32_t rounds_done = 0;
  if (blockIdx.x == 0 && tid == 0) S->status = kCseRunning;
  const unsigned long long barrier0 = vol_load64(&S->barriers);

  for (;;) {
    const int cur = round & 1, nxt = cur ^ 1;
    if (tid < 16) s_cnt[tid >> 1][tid & 1] = vol_load(&S->cnt[cur][tid >> 1][tid & 1]);
    if (tid >= 32 && tid < 40) s_emitted[tid - 32] = vol_load64(&S->emitted[cur][tid - 32]);
    __syncthreads();
    if (tid == 0) {
      uint32_t t = 0;
      unsigned long long nodes = 0;
      uint32_t drain = 0, widest = 0;
      for (int l = 0; l < 8; ++l) {
        unsigned long long lvl = 0;
        for (int h = 0; h < 2; ++h) {
          s_tstart[l][h] = t;
          t += (s_cnt[l][h] + TILE - 1) / TILE;
          lvl += s_cnt[l][h];
        }
        nodes += lvl;
        widest = max(widest, uint32_t(min(lvl, 0xFFFFFFFFull)));
        if (must_drain(s_emitted[l], lvl, max_words(a), a.ecap[l], a.esoft[l])) drain = 1;
      }
      // tiles per level, ascending, and the number of tiles scheduled before every breakpoint
      for (int l = 0; l < 8; ++l) s_lt[l] = (s_cnt[l][0] + TILE - 1) / TILE + (s_cnt[l][1] + TILE - 1) / TILE;
      for (int i = 0; i < 8; ++i) s_srt[i] = s_lt[i];
      for (int i = 1; i < 8; ++i) {                      // insertion sort of 8 values
        const uint32_t v = s_srt[i];
        int k = i - 1;
        while (k >= 0 && s_srt[k] > v) { s_srt[k + 1] = s_srt[k]; --k; }
        s_srt[k + 1] = v;
      }
      s_cum[0] = 0;
      for (int i = 0; i < 8; ++i) s_cum[i + 1] = s_cum[i] + (8 - i) * (s_srt[i] - (i ? s_srt[i - 1] : 0u));
      s_flags[0] = t;
      s_flags[1] = round_status(nodes, round, a.round_limit, false, a.use_narrow && widest <= a.narrow_enter,
                                nodes < a.min_nodes || nodes > a.max_nodes, drain);   // (leave: the host picks another kernel)
      if (blockIdx.x == 0 && s_flags[1] == kCseRunning) {
        S->visits += nodes;
        if (nodes > S->peak_frontier) S->peak_frontier = nodes;
      }
    }
    __syncthreads();
    const uint32_t total_tiles = s_flags[0];
    const uint32_t decision = s_flags[1];
    if (decision != kCseRunning) {
      if (blockIdx.x == 0 && tid == 0) { S->status = decision; S->round = round; S->barriers = barrier0 + rounds_done; }
      break;
    }
    if (blockIdx.x == 0 && tid < 8) {
      const int l = tid;
      if (s_cnt[l][0] + s_cnt[l][1] == 0) {
        S->cnt[nxt][(l + 1) & 7][0] = 0;
        S->cnt[nxt][(l + 1) & 7][1] = 0;
        S->emitted[nxt][l] = s_emitted[l];
      }
    }
    const uint32_t tag = round + 1;

    // ---- the tile being computed -------------------------------------------------------------
    uint32_t tile = blockIdx.x;
    uint32_t seq = 0;                                       // tiles of this round taken by this CTA so far
    bool have = tile < total_tiles;
    int l = 0, hh = 0, nv = 0;
    uint32_t tj = 0;                                        // position of the tile in its level's chain
    uint32_t ns[ITEMS], na[ITEMS], nb[ITEMS];
    uint64_t wa[ITEMS], wb[ITEMS], wc[ITEMS];
    // ---- the tile computed one iteration ago, waiting for its prefixes -----------------------
    bool p_valid = false, p_last = false;
    int p_l = 0;
    uint32_t p_desc = 0, p_first = 0, p_tz = 0, p_to = 0, p_te = 0;
    int buf = 0;

    // Schedule: the t-th tile handed out in a round is row r of the r-th "sweep" over the levels
    // that still have a tile r, so the gridDim tiles that run at the same time are spread
    // over all 8 chains instead of being consecutive links of one.  Returns the level, half,
    // this thread's nodes and the tile's position tj in its level's chain.
    auto locate_row = [&](uint32_t t, int& tl, uint32_t& r_out) {
      int seg = 0;
#pragma unroll
      for (int i = 1; i < 8; ++i)
        if (t >= s_cum[i]) seg = i;
      const uint32_t live = 8u - uint32_t(seg);                 // levels that have a tile in this row
      const uint32_t rel = t - s_cum[seg];
      const uint32_t r = (seg ? s_srt[seg - 1] : 0u) + rel / live;
      uint32_t pick = rel % live;
      tl = 0;
      bool found = false;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (!found && s_lt[k] > r) {
          if (pick == 0) { tl = k; found = true; } else --pick;
        }
      }
      r_out = r;
    };
    // every warp used to repeat locate_row for every tile (8 % of the kernel's instructions): the CTA's
    // tiles of the round are located once, cooperatively, and looked up afterwards
    {
      const uint32_t mine = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x - 1) / gridDim.x + 1 : 0u;
      const uint32_t fill = min(mine, uint32_t(SCHED_CAP));
      for (uint32_t i = tid; i < fill; i += CS_THREADS) {
        int tl;
        uint32_t r;
        locate_row(blockIdx.x + i * gridDim.x, tl, r);
        s_sched[i] = (uint32_t(tl) << 28) | r;
      }
    }
    __syncthreads();
    // seq = how many tiles of this round the CTA has taken before tile t
    auto locate = [&](uint32_t t, uint32_t seq, int& tl, int& th, int& tnv, uint32_t& to0, uint32_t& ttj) {
      uint32_t r;
      if (seq < uint32_t(SCHED_CAP)) { const uint32_t e = s_sched[seq]; tl = int(e >> 28); r = e & 0x0FFFFFFFu; }
      else locate_row(t, tl, r);
      ttj = r;
      const uint32_t th0 = (s_cnt[tl][0] + TILE - 1) / TILE;
      th = r < th0 ? 0 : 1;
      const uint32_t count = s_cnt[tl][th];
      to0 = (th ? r - th0 : r) * TILE + tid * ITEMS;
      tnv = to0 >= count ? 0 : int(min(uint32_t(ITEMS), count - to0));
    };
    auto load_nodes = [&](int tl, int th, int tnv, uint32_t to0) {
#pragma unroll
      for (int j = 0; j < ITEMS; ++j) ns[j] = na[j] = nb[j] = 0;
      if (tnv) {
        load_items<ITEMS>(a.fs[cur][tl], to0, th != 0, a.cap, ns);
        load_items<ITEMS>(a.fa[cur][tl], to0, th != 0, a.cap, na);
        load_items<ITEMS>(a.fb[cur][tl], to0, th != 0, a.cap, nb);
      }
    };
    auto gather = [&](int tl, int tnv) {
      const uint64_t* __restrict__ R = a.ranks[tl];
#pragma unroll
      for (int j = 0; j < ITEMS; ++j) {
        if (j < tnv) rank_words(R, ns[j], na[j], nb[j], wa[j], wb[j], wc[j]);
        else { wa[j] = wb[j] = wc[j] = 0; }
      }
    };

    if (have) {
      uint32_t o0;
      locate(tile, 0u, l, hh, nv, o0, tj);
      load_nodes(l, hh, nv, o0);
      gather(l, nv);
    }

    while (have || p_valid) {
      // ---- compute(i) ---------------------------------------------------------------------
      bool c_valid = false, c_last = false;
      int c_l = 0;
      uint32_t c_desc = 0, c_first = 0, c_tz = 0, c_to = 0, c_te = 0;
      if (have) {
        const uint32_t one_base = a.C[(l + 1) & 7];
        uint32_t fz = 0, fo = 0;
        uint32_t zs_[ITEMS], za0_[ITEMS], za1_[ITEMS], os_[ITEMS], oa0_[ITEMS], oa1_[ITEMS];
        uint32_t e0_[ITEMS], e1_[ITEMS], e2_[ITEMS], nw_[ITEMS];          // emitted words (see count_words)
        uint32_t nwords = 0;
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
          zs_[j] = za0_[j] = za1_[j] = os_[j] = oa0_[j] = oa1_[j] = e0_[j] = e1_[j] = e2_[j] = nw_[j] = 0;
          if (j < nv) {
            const CseStep r = cse_step(a, l, one_base, ns[j], na[j], nb[j], wa[j], wb[j], wc[j]);
            zs_[j] = r.zs; os_[j] = r.os;
            fz |= uint32_t(r.z) << j; za0_[j] = r.za; za1_[j] = r.zb;
            fo |= uint32_t(r.o) << j; oa0_[j] = r.oa; oa1_[j] = r.ob;
            nw_[j] = r.nw; e0_[j] = r.e0; e1_[j] = r.e1; e2_[j] = r.e2;
          }
        }
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) nwords += nw_[j];
        const uint64_t mine = uint64_t(__popc(fz)) | (uint64_t(__popc(fo)) << 21) | (uint64_t(nwords) << 42);
        uint64_t tile_tot;
        const uint64_t excl = block_exclusive_scan<uint64_t, CS_THREADS>(mine, s_scan, tile_tot);
        c_valid = true;
        c_l = l;
        c_first = s_tstart[l][0];                  // descriptors: one contiguous run per level
        c_desc = c_first + tj;
        c_last = tj + 1 == s_lt[l];
        c_tz = uint32_t(tile_tot) & 0x1FFFFFu;
        c_to = uint32_t(tile_tot >> 21) & 0x1FFFFFu;
        c_te = uint32_t(tile_tot >> 42) & 0x1FFFFFu;
        // publish the aggregates now; the prefixes are resolved one iteration later
        if (warp < 3 && lane == 0) {
          const uint32_t agg = uint32_t(tile_tot >> (21 * warp)) & 0x1FFFFFu;
          desc_store(a.desc + size_t(warp) * a.desc_tiles + c_desc,
                     desc_pack(tag, c_desc == c_first ? kDescPrefix : kDescAgg, agg));
        }
        {   // stage the outputs at their tile-local ordered positions
          WideStage<ITEMS, EW>& st = stage[buf];
          uint32_t lz = uint32_t(excl) & 0x1FFFFFu, lo_ = uint32_t(excl >> 21) & 0x1FFFFFu, le = uint32_t(excl >> 42) & 0x1FFFFFu;
#pragma unroll
          for (int j = 0; j < ITEMS; ++j) {
            if (fz >> j & 1u) { st.zs[lz] = zs_[j]; st.za[lz] = za0_[j]; st.zb[lz] = za1_[j]; ++lz; }
            if (fo >> j & 1u) { st.os[lo_] = os_[j]; st.oa[lo_] = oa0_[j]; st.ob[lo_] = oa1_[j]; ++lo_; }
            if (nw_[j]) {
              put_words(st.e + le, nw_[j], e0_[j], e1_[j], e2_[j], nb[j], na[j] + nb[j]);
              le += nw_[j];
            }
          }
        }
      }
      // ---- load(i+1): the node registers of tile i are dead from here on ----------------------
      const uint32_t next = tile + gridDim.x;
      const bool have_next = have && next < total_tiles;
      int l2 = 0, hh2 = 0, nv2 = 0;
      uint32_t tj2 = 0;
      if (have_next) {
        uint32_t o02;
        locate(next, ++seq, l2, hh2, nv2, o02, tj2);
        load_nodes(l2, hh2, nv2, o02);
      }
      // ---- resolve(i-1) --------------------------------------------------------------------------
      if (p_valid && warp < 3) {
        const uint32_t agg = warp == 0 ? p_tz : (warp == 1 ? p_to : p_te);
        uint32_t pre = 0;
        if (p_desc != p_first)
          pre = lookback_resolve_wide<4>(a.desc + size_t(warp) * a.desc_tiles, p_desc, p_first, tag, agg, &S->err);
        if (lane == 0) s_prefix[warp] = pre;
      }
      __syncthreads();          // staged outputs (both buffers) and prefixes are visible to everyone
      // ---- gather(i+1) ----------------------------------------------------------------------------
      if (have_next) gather(l2, nv2);
      // ---- flush(i-1) -------------------------------------------------------------------------------
      if (p_valid) {
        const WideStage<ITEMS, EW>& st = stage[buf ^ 1];
        const int ln = (p_l + 1) & 7;
        const uint32_t pz = s_prefix[0], po = s_prefix[1];
        const unsigned long long pe = s_emitted[p_l] + s_prefix[2];
        uint32_t* __restrict__ gs = a.fs[nxt][ln];
        uint32_t* __restrict__ ga = a.fa[nxt][ln];
        uint32_t* __restrict__ gb = a.fb[nxt][ln];
        for (uint32_t j = tid; j < p_tz; j += CS_THREADS) {
          const uint32_t at = pz + j;
          if (at < a.cap) { gs[at] = st.zs[j]; ga[at] = st.za[j]; gb[at] = st.zb[j]; }
        }
        for (uint32_t j = tid; j < p_to; j += CS_THREADS) {
          const uint32_t ord = po + j;                 // one-half is stored back to front
          if (ord < a.cap) { const uint32_t at = a.cap - 1 - ord; gs[at] = st.os[j]; ga[at] = st.oa[j]; gb[at] = st.ob[j]; }
        }
        if (pe + p_te <= a.ecap[p_l]) {
          uint32_t* __restrict__ ew = a.emit[p_l] + pe;
          for (uint32_t w = tid; w < p_te; w += CS_THREADS) ew[w] = st.e[w];
        }
        if (p_last && tid == 0) {
          S->cnt[nxt][ln][0] = pz + p_tz;
          S->cnt[nxt][ln][1] = po + p_to;
          S->emitted[nxt][p_l] = pe + p_te;
          if (uint64_t(pz) + p_tz + po + p_to > a.cap) atomicExch(&S->status, uint32_t(kCseOverflow));
        }
      }
      __syncthreads();          // buffer buf^1, s_prefix and s_scan are free again
      p_valid = c_valid; p_last = c_last; p_l = c_l; p_desc = c_desc; p_first = c_first;
      p_tz = c_tz; p_to = c_to; p_te = c_te;
      buf ^= 1;
      tile = next; have = have_next; l = l2; hh = hh2; nv = nv2; tj = tj2;
    }

    grid_barrier(S, barrier0 + rounds_done, round);
    ++round;
    ++rounds_done;
    if (vol_load(&S->status) != kCseRunning || vol_load(&S->err) != 0) {
      if (blockIdx.x == 0 && tid == 0) { S->round = round; S->barriers = barrier0 + rounds_done; }
      break;
    }
  }
}

}  // namespace bce
