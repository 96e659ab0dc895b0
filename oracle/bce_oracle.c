/*
 * oracle/bce_oracle.c -- TEST INFRASTRUCTURE, not product code (see bce_oracle.h).
 *
 * Plain-C restatement of the reference front end (rotate, BWT, wavelet matrix,
 * CSE level loop) and of the host-side archive writer, each function citing the
 * lines of /root/reference/bce.cpp it follows.  Queues are flat arrays of
 * absolute positions instead of the reference's Elias-gamma pArray (:226-356):
 * the gamma coding is a memory optimisation and is not visible in the archive.
 */
#include "bce_oracle.h"
#include "divsufsort.h"

#include <stdlib.h>
#include <string.h>

void bceo_free(void *p) { free(p); }

/* ------------------------------------------------------------------ */
/* File::rotate, bce.cpp:858-894                                       */
/* ------------------------------------------------------------------ */
uint32_t bceo_least_rotation(const uint8_t *T, size_t n) {
  /* two candidates i < j and a match length k; the loser jumps past the
   * mismatch (:869-882).  Indices wrap with at most one subtraction (:859-862). */
  size_t i = 0, j = 1;
  while (j < n) {
    size_t k = 0;
    for (;;) {
      size_t a = i + k, b = j + k;
      if (a >= n) a -= n;
      if (b >= n) b -= n;
      if (!(T[a] == T[b] && k < n - 1)) break;       /* :871 */
      ++k;
    }
    size_t a = i + k, b = j + k;
    if (a >= n) a -= n;
    if (b >= n) b -= n;
    if (T[a] <= T[b]) {                              /* :873-874 */
      j += k + 1;
    } else {                                         /* :875-881 */
      i += k + 1;
      if (i < j) { i = j; ++j; }
      else j = i + 1;
    }
  }
  return (uint32_t)i;
}

/* smallest p dividing n such that T is p-periodic (n if T is primitive) */
static uint32_t smallest_full_period(const uint8_t *T, uint32_t n) {
  uint32_t *pi = (uint32_t *)malloc((size_t)n * sizeof(uint32_t));
  if (!pi) return n;
  pi[0] = 0;
  for (uint32_t q = 1, k = 0; q < n; ++q) {
    while (k > 0 && T[k] != T[q]) k = pi[k - 1];
    if (T[k] == T[q]) ++k;
    pi[q] = k;
  }
  uint32_t p = n - pi[n - 1];
  free(pi);
  return (n % p == 0) ? p : n;
}

static int cmp_u32(const void *a, const void *b) {
  uint32_t x = *(const uint32_t *)a, y = *(const uint32_t *)b;
  return (x > y) - (x < y);
}

/* ------------------------------------------------------------------ */
/* File::rotate + File::bwt, bce.cpp:858-910                           */
/* ------------------------------------------------------------------ */
int bceo_bwt(const uint8_t *T, uint32_t n, uint8_t *L, uint32_t *offset, uint32_t *SA_out) {
  if (!T || !L || n == 0) return -1;
  uint32_t i = bceo_least_rotation(T, n);
  if (offset) *offset = i;
  /* :884  rotate left by i+1: buffer = R[1..n-1] R[0], R = least rotation */
  uint8_t *buf = (uint8_t *)malloc((size_t)n);
  if (!buf) return -2;
  uint32_t cut = (i + 1) % n;
  memcpy(buf, T + cut, (size_t)(n - cut));
  memcpy(buf + (n - cut), T, (size_t)cut);
  /* :901  BWT of the first n-1 bytes in place, primary index p */
  saidx_t p = divbwt(buf, buf, NULL, (saidx_t)(n - 1));
  if (p < 0) { free(buf); return -2; }
  /* :902  splice the last byte (R[0]) in at position p */
  uint8_t last = buf[n - 1];
  memmove(buf + p + 1, buf + p, (size_t)(n - 1 - (uint32_t)p));
  buf[p] = last;
  memcpy(L, buf, (size_t)n);

  if (SA_out) {
    /* row 0 is R itself; row r>=1 is the (r-1)-th smallest suffix of R[1..n-1] */
    SA_out[0] = i;
    if (n > 1) {
      memcpy(buf, T + cut, (size_t)(n - cut));
      memcpy(buf + (n - cut), T, (size_t)cut);
      saidx_t *sa = (saidx_t *)malloc((size_t)(n - 1) * sizeof(saidx_t));
      if (!sa || divsufsort(buf, sa, (saidx_t)(n - 1)) != 0) { free(sa); free(buf); return -2; }
      for (uint32_t r = 1; r < n; ++r)
        SA_out[r] = (uint32_t)(((uint64_t)i + 1u + (uint32_t)sa[r - 1]) % n);
      free(sa);
      uint32_t p0 = smallest_full_period(T, n);
      if (p0 < n) {                       /* identical rotations: order them by index */
        uint32_t reps = n / p0;
        for (uint32_t r = 0; r < n; r += reps) qsort(SA_out + r, reps, sizeof(uint32_t), cmp_u32);
      }
    }
  }
  free(buf);
  return 0;
}

/* ------------------------------------------------------------------ */
/* Rank::get<1>, bce.cpp:147-151                                       */
/* ------------------------------------------------------------------ */
uint32_t bceo_rank1(const uint64_t *rank, uint32_t index) {
  uint64_t w = rank[index / 32];
  uint32_t below = (uint32_t)(w >> 32) & (uint32_t)((1ull << (index % 32)) - 1);
  return (uint32_t)w + (uint32_t)__builtin_popcount(below);
}
static inline uint32_t rank0(const uint64_t *rank, uint32_t index) {   /* :216-219 */
  return index - bceo_rank1(rank, index);
}
static inline uint32_t bit_at(const uint64_t *rank, uint32_t index) {  /* :196-198 */
  return (uint32_t)(rank[index / 32] >> (index % 32 + 32)) & 1u;
}

/* ------------------------------------------------------------------ */
/* RankFile ctor, bce.cpp:944-972; Rank::build :138-145                */
/* ------------------------------------------------------------------ */
void bceo_wavelet(const uint8_t *L, uint32_t n, uint64_t *const ranks[8]) {
  size_t words = bceo_rank_words(n);
  for (int j = 0; j < 8; ++j) memset(ranks[j], 0, words * sizeof(uint64_t));

  /* next[j][ctx] = write cursor of level j for bytes whose low j bits are ctx:
   * exclusive prefix (numeric ctx order) of the counts (:947-960); on the stack, so that threads can build
   * wavelet matrices side by side */
  uint32_t next[8][128];
  uint32_t hist[256];
  memset(hist, 0, sizeof hist);
  for (uint32_t p = 0; p < n; ++p) hist[L[p]]++;
  for (int j = 0; j < 8; ++j) {
    uint32_t groups = 1u << j, run = 0;
    for (uint32_t ctx = 0; ctx < groups; ++ctx) {
      uint32_t c = 0;
      for (uint32_t v = ctx; v < 256; v += groups) c += hist[v];
      next[j][ctx] = run;
      run += c;
    }
  }
  /* :962-968  bit j of every byte goes to level j at its context's cursor */
  for (uint32_t p = 0; p < n; ++p) {
    uint32_t chr = L[p];
    for (int j = 0; j < 8; ++j) {
      uint32_t ctx = chr & ((1u << j) - 1);
      uint32_t at = next[j][ctx]++;
      ranks[j][at / 32] |= (uint64_t)((chr >> j) & 1u) << (at % 32);
    }
  }
  /* :138-145  word = bits << 32 | ones before this word */
  for (int j = 0; j < 8; ++j) {
    uint32_t run = 0;
    for (size_t w = 0; w < words; ++w) {
      uint64_t b = ranks[j][w];
      ranks[j][w] = (b << 32) | run;
      run += (uint32_t)__builtin_popcountll(b);
    }
  }
}

/* ------------------------------------------------------------------ */
/* BCE::encode roots :1124-1130 and BCE::code(mode=1) :1236-1373       */
/* ------------------------------------------------------------------ */
typedef struct { uint32_t *v; size_t len, cap; } nodevec;     /* triples (s, x0, x1) */

static int nv_push(nodevec *q, uint32_t s, uint32_t a, uint32_t b) {
  if (q->len + 3 > q->cap) {
    size_t nc = q->cap ? q->cap * 2 : 1024;
    uint32_t *nv = (uint32_t *)realloc(q->v, nc * sizeof(uint32_t));
    if (!nv) return -1;
    q->v = nv; q->cap = nc;
  }
  q->v[q->len++] = s; q->v[q->len++] = a; q->v[q->len++] = b;
  return 0;
}

static int emit(bceo_cse_result *r, int lvl, uint32_t sym, uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs) {
  if (r->count[lvl] == r->cap[lvl]) {
    size_t nc = r->cap[lvl] ? r->cap[lvl] * 2 : 4096;
    bceo_tuple *nt = (bceo_tuple *)realloc(r->tuples[lvl], nc * sizeof(bceo_tuple));
    if (!nt) return -1;
    r->tuples[lvl] = nt; r->cap[lvl] = nc;
  }
  bceo_tuple *t = &r->tuples[lvl][r->count[lvl]++];
  t->sym = sym; t->k = k; t->c1 = c1; t->c2 = c2; t->cs = cs;
  return 0;
}

void bceo_cse_free(bceo_cse_result *r) {
  if (!r) return;
  for (int i = 0; i < 8; ++i) { free(r->tuples[i]); r->tuples[i] = NULL; r->count[i] = r->cap[i] = 0; }
}

int bceo_cse(const uint64_t *const ranks[8], uint32_t n, bceo_cse_result *out) {
  memset(out, 0, sizeof *out);
  /* cur[i][0/1]: nodes of level i in the zero / one half, ascending position;
   * nxt[i][0/1]: zero / one children produced by level i this round (:1237) */
  nodevec cur[8][2], nxt[8][2];
  memset(cur, 0, sizeof cur);
  memset(nxt, 0, sizeof nxt);
  int rc = 0;

  for (int i = 0; i < 8; ++i) {
    out->C[i] = rank0(ranks[(i + 7) % 8], n);                       /* :1128 */
    if (out->C[i] && n - out->C[i])                                 /* :1239-1240 */
      if (nv_push(&cur[i][0], 0, out->C[i], n - out->C[i])) rc = -2;
  }

  int again = rc == 0;
  while (again) {                                                   /* :1246 */
    again = 0;
    uint64_t frontier = 0;
    for (int i = 0; i < 8 && rc == 0; ++i) {                        /* :1252 */
      const uint64_t *R = ranks[i];
      const uint32_t child_one_base = out->C[(i + 1) % 8];          /* :1259 of the next level */
      for (int j = 0; j < 2 && rc == 0; ++j) {                      /* :1256 */
        const nodevec *q = &cur[i][j];
        frontier += q->len / 3;
        for (size_t t = 0; t < q->len && rc == 0; t += 3) {         /* :1261 */
          out->visits[i]++;
          uint32_t s = q->v[t], x0 = q->v[t + 1], x1 = q->v[t + 2];
          uint32_t x = x0 + x1;
          uint32_t s1 = bceo_rank1(R, s);                           /* :1265 */
          uint32_t n1x = bceo_rank1(R, s + x) - s1;                 /* :1271 */
          uint32_t s0 = s - s1;                                     /* :1272 */
          if (n1x == 0) {                                           /* :1274-1279 */
            if (nv_push(&nxt[i][0], s0, x0, x1)) rc = -2;
            continue;
          }
          uint32_t n0x = x - n1x;                                   /* :1281 */
          if (n0x == 0) {                                           /* :1282-1287 */
            if (nv_push(&nxt[i][1], child_one_base + s1, x0, x1)) rc = -2;
            continue;
          }
          /* :1290-1294  feasible range of n0x0 */
          uint32_t lo = x0 > n1x ? x0 - n1x : 0;
          uint32_t hi = x0 - (n1x > x1 ? n1x - x1 : 0);
          uint32_t n0x0 = lo;                                       /* :1297 */
          if (hi != lo) {                                           /* :1299-1302 */
            n0x0 = rank0(R, s + x0) - s0;
            if (emit(out, i, n0x0 - lo, hi - lo + 1, n0x, x1, x)) rc = -2;
          }
          uint32_t n0x1 = n0x - n0x0;                               /* :1337 */
          if (n0x0 && n0x1)
            if (nv_push(&nxt[i][0], s0, n0x0, n0x1)) rc = -2;       /* :1338-1341 */
          uint32_t n1x1 = x1 - n0x1;                                /* :1343 */
          uint32_t n1x0 = n1x - n1x1;                               /* :1344 */
          if (n1x0 && n1x1)
            if (nv_push(&nxt[i][1], child_one_base + s1, n1x0, n1x1)) rc = -2;  /* :1345-1348 */
        }
      }
    }
    if (frontier > out->peak_frontier) out->peak_frontier = frontier;
    out->rounds++;
    /* :1361-1370  children of level i become the queues of level (i+1)%8 */
    for (int i = 0; i < 8; ++i) { cur[i][0].len = 0; cur[i][1].len = 0; }
    for (int i = 0; i < 8; ++i) {
      int d = (i + 1) % 8;
      for (int j = 0; j < 2; ++j) {
        nodevec tmp = cur[d][j]; cur[d][j] = nxt[i][j]; nxt[i][j] = tmp;
        nxt[i][j].len = 0;
        if (cur[d][j].len) again = 1;
      }
    }
    if (rc) break;
  }
  for (int i = 0; i < 8; ++i)
    for (int j = 0; j < 2; ++j) { free(cur[i][j].v); free(nxt[i][j].v); }
  if (rc) bceo_cse_free(out);
  return rc;
}

/* ------------------------------------------------------------------ */
/* AdaptiveCoder<31> encode side, bce.cpp:484-724; VCoder :362-378     */
/* ------------------------------------------------------------------ */
static const uint8_t k_default_cfg[9 * 32] = {                       /* :713-724 */
  0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,0,
  0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,0,
  0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,3,3,3,3,0,
  0,0,5,5,5,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,0,
  0,0,5,5,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0,
  0,0,5,5,4,4,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0,
  0,0,5,4,4,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,0,
  0,0,4,4,4,4,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,3,2,2,2,2,2,2,0,
  0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0
};
const uint8_t *bceo_default_config(void) { return k_default_cfg; }

typedef struct {
  uint64_t lo, hi;                 /* l_, h_  :644-645 */
  uint16_t *out; size_t len, cap;  /* data_   :649 */
  uint32_t off[32];                /* off_    :650 */
  uint8_t *stat;                   /* stat_   :651 */
  int oom;
} acoder;

static void ac_put(acoder *c, uint16_t w) {
  if (c->len == c->cap) {
    size_t nc = c->cap ? c->cap * 2 : 1024;
    uint16_t *no = (uint16_t *)realloc(c->out, nc * sizeof(uint16_t));
    if (!no) { c->oom = 1; return; }
    c->out = no; c->cap = nc;
  }
  c->out[c->len++] = w;
}
static void ac_shift_out(acoder *c) {                                /* :655-661 */
  while (((c->hi ^ c->lo) >> 48) == 0) {
    ac_put(c, (uint16_t)(c->hi >> 48));
    c->lo <<= 16;
    c->hi = (c->hi << 16) | 0xFFFFu;
  }
}
static void ac_restart_if_narrow(acoder *c, uint64_t total) {        /* :520-525, :541-546 */
  if (c->hi - c->lo < total) {
    for (int i = 0; i < 4; ++i) ac_put(c, (uint16_t)(c->lo >> (48 - 16 * i)));
    c->lo = 0; c->hi = ~0ull;
  }
}
static void ac_uniform(acoder *c, uint32_t s, uint32_t k) {          /* :538-553 */
  ac_restart_if_narrow(c, k);
  uint64_t step = (c->hi - c->lo) / k;
  c->lo += step * s;
  c->hi = c->lo + step - 1;
  ac_shift_out(c);
}
static void ac_adaptive(acoder *c, uint32_t s, uint32_t k, uint32_t c1, uint32_t c2, uint32_t cs) {
  while (k > 31) {                                                   /* :507-510 */
    ac_uniform(c, s & 1, 2);
    k = (k + (~s & 1)) >> 1;
    s >>= 1;
  }
  uint32_t off = c->off[k];                                          /* :671-677 */
  uint32_t bits = off >> 24;
  uint32_t ctx = (((uint32_t)(c1 << bits) / cs) << bits) | ((uint32_t)(c2 << bits) / cs);
  uint8_t *row = c->stat + (off & 0x00FFFFFFu) + (size_t)ctx * k;
  uint32_t below = s, total = k;                                     /* :514-518 */
  for (uint32_t i = 0; i < s; ++i) below += row[i];
  for (uint32_t i = 0; i < k; ++i) total += row[i];
  ac_restart_if_narrow(c, total);
  uint64_t step = (c->hi - c->lo) / total;                           /* :527-529 */
  c->lo += step * below;
  c->hi = c->lo + step * ((uint64_t)row[s] + 1) - 1;
  if (++row[s] == 0xFF)                                              /* :531-533 */
    for (uint32_t i = 0; i < k; ++i) row[i] >>= 1;
  ac_shift_out(c);
}
static void ac_setv(acoder *c, uint32_t v) {                         /* :364-370 */
  while (v) { ac_uniform(c, v & 1, 3); v >>= 1; }
  ac_uniform(c, 2, 3);
}
static void ac_flush(acoder *c) {                                    /* :610-615 */
  ac_shift_out(c);
  uint32_t bits = (uint32_t)__builtin_clzll(c->lo ^ c->hi) + 1;
  ac_put(c, (uint16_t)((c->hi >> (64 - bits)) << (16 - bits)));
}
static int ac_init(acoder *c, int id, const uint8_t *cfg) {          /* :491-493, :679-710 */
  memset(c, 0, sizeof *c);
  c->lo = 0; c->hi = ~0ull;
  const uint8_t *row = cfg + 32 * ((id < 0 || id > 7) ? 8 : id);     /* :683-684 */
  uint32_t last = 0;
  for (int i = 0; i < 32; ++i) {                                     /* :685-691 */
    uint32_t b = row[i];
    ac_uniform(c, b != last, 2);
    if (b != last) ac_uniform(c, b, 6);
    last = b;
  }
  uint32_t start = 0;                                                /* :700-705 */
  for (uint32_t k = 2; k < 32; ++k) {
    c->off[k] = start | ((uint32_t)row[k] << 24);
    start += k << (row[k] * 2);
  }
  c->stat = (uint8_t *)calloc(start ? start : 1, 1);
  return c->stat ? 0 : -2;
}
static void ac_destroy(acoder *c) { free(c->out); free(c->stat); memset(c, 0, sizeof *c); }

/* ------------------------------------------------------------------ */
/* BCE::encode, bce.cpp:1117-1167 (coder side)                         */
/* ------------------------------------------------------------------ */
int bceo_encode_archive(const bceo_cse_result *cse, uint32_t n, uint32_t offset,
                        const uint8_t *cfg, uint16_t **words, size_t *nwords) {
  if (!cfg) cfg = k_default_cfg;
  acoder st[8], hdr;
  memset(st, 0, sizeof st);
  memset(&hdr, 0, sizeof hdr);
  int rc = 0;
  uint32_t total = 0;
  for (int i = 0; i < 8 && rc == 0; ++i) {
    rc = ac_init(&st[i], i, cfg);                                    /* :1124 */
    if (rc) break;
    ac_uniform(&st[i], cse->C[i], n + 1);                            /* :1129 */
    for (size_t t = 0; t < cse->count[i]; ++t) {                     /* :1302 */
      const bceo_tuple *u = &cse->tuples[i][t];
      ac_adaptive(&st[i], u->sym, u->k, u->c1, u->c2, u->cs);
    }
    ac_flush(&st[i]);                                                /* :1136 */
    total += (uint32_t)st[i].len;                                    /* :1137 */
    if (st[i].oom) rc = -2;
  }
  if (rc == 0) rc = ac_init(&hdr, -1, cfg);                          /* :1141 */
  if (rc == 0) {
    ac_setv(&hdr, n);                                                /* :1142 */
    ac_uniform(&hdr, offset, n + 1);                                 /* :1143 */
    ac_setv(&hdr, total);                                            /* :1144 */
    uint32_t left = total;
    for (int i = 0; i < 7; ++i) {                                    /* :1145-1148 */
      ac_uniform(&hdr, (uint32_t)st[i].len, left + 1);
      left -= (uint32_t)st[i].len;
    }
    ac_flush(&hdr);                                                  /* :1149 */
    if (hdr.oom) rc = -2;
  }
  if (rc == 0) {
    size_t nw = 1 + hdr.len + total;                                 /* :1152-1157 */
    uint16_t *w = (uint16_t *)malloc(nw * sizeof(uint16_t));
    if (!w) rc = -2;
    else {
      size_t at = 0;
      w[at++] = (uint16_t)hdr.len;
      memcpy(w + at, hdr.out, hdr.len * sizeof(uint16_t)); at += hdr.len;
      for (int i = 0; i < 8; ++i) { memcpy(w + at, st[i].out, st[i].len * sizeof(uint16_t)); at += st[i].len; }
      *words = w; *nwords = nw;
    }
  }
  for (int i = 0; i < 8; ++i) ac_destroy(&st[i]);
  ac_destroy(&hdr);
  return rc;
}

int bceo_compress(const uint8_t *T, uint32_t n, const uint8_t *cfg,
                  uint16_t **words, size_t *nwords) {
  if (n == 0) return -1;
  size_t rw = bceo_rank_words(n);
  uint8_t *L = (uint8_t *)malloc(n);
  uint64_t *store = (uint64_t *)malloc(8 * rw * sizeof(uint64_t));
  if (!L || !store) { free(L); free(store); return -2; }
  uint64_t *ranks[8];
  for (int j = 0; j < 8; ++j) ranks[j] = store + (size_t)j * rw;
  uint32_t offset = 0;
  int rc = bceo_bwt(T, n, L, &offset, NULL);
  bceo_cse_result cse;
  memset(&cse, 0, sizeof cse);
  if (rc == 0) {
    bceo_wavelet(L, n, ranks);
    rc = bceo_cse((const uint64_t *const *)ranks, n, &cse);
  }
  if (rc == 0) rc = bceo_encode_archive(&cse, n, offset, cfg, words, nwords);
  bceo_cse_free(&cse);
  free(L); free(store);
  return rc;
}

/* ------------------------------------------------------------------ */
/* unbwt::bitwise, bce.cpp:999-1038                                    */
/* ------------------------------------------------------------------ */
void bceo_unbwt_bitwise(const uint64_t *const ranks[8], uint32_t offset, uint32_t n, uint8_t *out) {
  uint32_t zeros[8];
  for (int j = 0; j < 8; ++j) zeros[j] = rank0(ranks[j], n);        /* :1006-1015 */
  uint64_t s = 0;
  for (uint64_t i = n; i-- > 0;) {                                   /* :1019 */
    uint32_t chr = 0;
    for (int j = 0; j < 8; ++j) {                                    /* :1021-1027 */
      uint32_t b = bit_at(ranks[j], (uint32_t)s);
      chr |= b << j;
      s = b ? zeros[j] + bceo_rank1(ranks[j], (uint32_t)s) : rank0(ranks[j], (uint32_t)s);
    }
    out[(i + offset) % n] = (uint8_t)chr;                            /* :1028 */
  }
}

/* first half of unbwt::bytewise, bce.cpp:1050-1085 */
void bceo_wavelet_to_bytes(const uint64_t *const ranks[8], uint32_t n, uint8_t *L) {
  uint32_t zeros[8];
  for (int j = 0; j < 8; ++j) zeros[j] = rank0(ranks[j], n);        /* :1052-1061 */
  /* cursor[(1<<j)|ctx] = position in level j of the next byte whose low j bits are ctx.
   * The reference restarts these per chunk (:1066-1077); one chunk from 0 is the same. */
  uint32_t cursor[256];
  memset(cursor, 0, sizeof cursor);
  cursor[1] = 0;
  for (int j = 0; j < 7; ++j)
    for (uint32_t ctx = 0; ctx < (1u << j); ++ctx) {
      uint32_t e = cursor[(1u << j) | ctx];
      cursor[(2u << j) | ctx] = rank0(ranks[j], e);
      cursor[(3u << j) | ctx] = zeros[j] + bceo_rank1(ranks[j], e);
    }
  for (uint32_t p = 0; p < n; ++p) {                                 /* :1079-1084 */
    uint32_t chr = 0;
    for (int j = 0; j < 8; ++j)
      chr |= bit_at(ranks[j], cursor[(1u << j) | chr]++) << j;
    L[p] = (uint8_t)chr;
  }
}

/* unbwt::bytewise, bce.cpp:1043-1103 */
int bceo_unbwt_bytewise(const uint64_t *const ranks[8], uint32_t offset, uint32_t n, uint8_t *out) {
  uint8_t *L = (uint8_t *)malloc(n ? n : 1);
  if (!L) return -2;
  bceo_wavelet_to_bytes(ranks, n, L);
  if (inverse_bw_transform(L, L, NULL, (saidx_t)n, 1) != 0 && n > 1) { free(L); return -1; }  /* :1091 */
  /* :1093 rotate right by offset */
  for (uint32_t p = 0; p < n; ++p) out[(p + offset) % n] = L[p];
  free(L);
  return 0;
}

/* see bce_oracle.h: the per-stream sums of oracle/ref_tap.cpp (TapStore) over a batch of calls */
void bceo_call_checksum(const uint32_t *t, size_t count, uint64_t first, uint64_t out[2]) {
  const uint64_t A = 0x9E3779B97F4A7C15ull;
  uint64_t sum = 0, wsum = 0;
  for (size_t j = 0; j < count; ++j, t += 5) {
    const uint64_t h = ((((uint64_t)t[0] * A + t[1]) * A + t[2]) * A + t[3]) * A + t[4];
    sum += h;
    wsum += h * (2 * (first + j) + 1);
  }
  out[0] = sum;
  out[1] = wsum;
}

void bceo_word_checksum(const uint32_t *w, size_t count, uint64_t first, uint64_t out[2]) {
  uint64_t sum = 0, wsum = 0;
  for (size_t j = 0; j < count; ++j) {
    sum += w[j];
    wsum += (uint64_t)w[j] * (2 * (first + j) + 1);
  }
  out[0] = sum;
  out[1] = wsum;
}
