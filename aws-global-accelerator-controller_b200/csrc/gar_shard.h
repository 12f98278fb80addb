// gar_shard.h — ONE cluster sharded by key hash across ranks (SURVEY.md §8 row e, BASELINE configs[3]:
// "10^7 objects sharded by key-hash across 8xB200 with one NCCL all-to-all").
//
// Every rank starts with an arbitrary contiguous slice of each list (the packer just cuts the lister output and the
// paginated AWS lists into n_ranks ranges; include/garecon.h "sharded mode").  The diff is a join DAG over several keys,
// so rows are re-homed on the device:
//
//   round 1 (the all-to-all): every row travels to the shard its OWN key hashes to
//        objects                               -> home(key_hash_kinded(kind, "ns/name"))
//        accelerators of this cluster (+tags, listeners, port ranges, endpoint groups, endpoints)
//                                              -> home(owner tag key)           ["own" rows: owner lookups, orphans]
//        owner values (TXT) with their record  -> home(owner key inside the value)
//        alias records                         -> every home an owner value under the same (zone, name) goes to
//                                                 (the TXT-join-A on (zone, name) is local: whole zones stay together)
//      and, for the two lookups keyed by something the OBJECT does not own (its load balancer's hostname):
//        load balancers                        -> dir(key_hash_lb(region, name))
//        accelerator stubs (row + tags)        -> dir(directory key of the target-hostname tag)
//        one probe per lbIngress hostname      -> dir(directory key of the hostname), carrying home(object)
//   round 2 (answers, small): each directory shard resolves its probes against the rows it received (first row wins,
//      global order) and forwards the matching LB row / the first two by-hostname accelerators to the probe's home.
//
// After round 2 every rank holds a SELF-CONTAINED sub-snapshot (own objects + everything their decisions read) and runs
// the ordinary single-GPU pipeline on it; ops and statuses come back with GLOBAL row ids.  Accelerators that arrived as
// answers are "guest" rows: they serve by-target-hostname lookups only (Work::acc_guest_from).
//
// The exchange itself is the host's job (torch.distributed all_to_all_single over NCCL/NVLink in ranks.py): this file
// plans, packs one contiguous blob per destination, and merges the received blobs.  Same text runs in tests/hostsim.
//
// Backend additions:  void *shard_alloc(int arena, size_t bytes);  void shard_reset(int arena);
//                     void copy_bytes(void *dst, const void *src, size_t n);
#pragma once

#include "gar_pipeline.h"

#if defined(__CUDA_ARCH__)
#define GAR_ATOMIC_OR(p, v) atomicOr((p), (v))
#else
#define GAR_ATOMIC_OR(p, v) (*(p) |= (v))
#endif

constexpr int SH_MAX_RANKS = GAR_SHARD_MAX_RANKS;
constexpr int SH_MAX_SEGS = 2 * SH_MAX_RANKS;
enum ShLevel { L_OBJ, L_ANN, L_LBI, L_PORT, L_ACC, L_TAG, L_LIS, L_PR, L_EG, L_EP, L_REC, L_VAL, L_ZONE, L_LB, L_STUB, L_STUBTAG, L_PROBE, L_NLEVELS };
static_assert(2 * L_NLEVELS + 1 <= GAR_SHARD_META_WORDS, "meta row too small");
constexpr int SH_MAX_STR = 4, SH_MAX_U8 = 3, SH_MAX_U32 = 1, SH_MAX_CHILD = 3;
enum { SH_ARENA_PLAN = 0, SH_ARENA_DIR = 1, SH_ARENA_HOME = 2 };
constexpr u32 SH_DROP = 255;    // destination of a row nobody needs
constexpr u32 SH_FOLLOW = 254;  // child_dest value: the child goes wherever its parent goes

struct LevelSchema {
  int n_str, n_u8, n_u32, has_gid, n_child;
  int child[SH_MAX_CHILD];
};
// columns per level (order = the order of the fields in include/garecon.h)
static const LevelSchema SH_SCHEMA[L_NLEVELS] = {
    /* OBJ     */ {2, 3, 1, 1, 3, {L_ANN, L_LBI, L_PORT}},  // "ns/name" key, ingress_class | kind, spec_type, flags | ns_len
    /* ANN     */ {2, 0, 0, 0, 0, {0, 0, 0}},
    /* LBI     */ {1, 0, 0, 0, 0, {0, 0, 0}},
    /* PORT    */ {1, 0, 1, 0, 0, {0, 0, 0}},               // proto | number
    /* ACC     */ {2, 1, 0, 1, 2, {L_TAG, L_LIS, 0}},       // name, dns | enabled
    /* TAG     */ {2, 0, 0, 0, 0, {0, 0, 0}},
    /* LIS     */ {0, 1, 0, 1, 2, {L_PR, L_EG, 0}},         // proto
    /* PR      */ {0, 0, 1, 0, 0, {0, 0, 0}},
    /* EG      */ {0, 0, 0, 1, 1, {L_EP, 0, 0}},
    /* EP      */ {1, 0, 0, 0, 0, {0, 0, 0}},
    /* REC     */ {2, 2, 1, 1, 1, {L_VAL, 0, 0}},           // name, alias_dns | type, has_alias | zone
    /* VAL     */ {1, 0, 0, 1, 0, {0, 0, 0}},
    /* ZONE    */ {1, 0, 0, 0, 0, {0, 0, 0}},
    /* LB      */ {4, 1, 0, 1, 0, {0, 0, 0}},               // region, name, dns, arn | state
    /* STUB    */ {2, 1, 0, 1, 1, {L_STUBTAG, 0, 0}},       // an accelerator row without its listeners
    /* STUBTAG */ {2, 0, 0, 0, 0, {0, 0, 0}},
    /* PROBE   */ {1, 0, 1, 0, 0, {0, 0, 0}},               // hostname | home shard
};

// byte offsets of one level's columns inside a blob (all 16-byte aligned)
struct LevelLayout {
  u64 str[SH_MAX_STR], u8c[SH_MAX_U8], u32c[SH_MAX_U32], gid, cnt[SH_MAX_CHILD], slab, end;
};
inline u64 sh_align(u64 x) { return (x + 15) & ~(u64)15; }
inline LevelLayout level_layout(int lvl, u64 base, u64 n, u64 slab_bytes) {
  const LevelSchema &S = SH_SCHEMA[lvl];
  LevelLayout L{};
  u64 p = base;
  for (int c = 0; c < S.n_str; c++) { L.str[c] = p; p = sh_align(p + 8 * n); }
  for (int c = 0; c < S.n_u8; c++) { L.u8c[c] = p; p = sh_align(p + n); }
  for (int c = 0; c < S.n_u32; c++) { L.u32c[c] = p; p = sh_align(p + 4 * n); }
  if (S.has_gid) { L.gid = p; p = sh_align(p + 4 * n); }
  for (int c = 0; c < S.n_child; c++) { L.cnt[c] = p; p = sh_align(p + 4 * n); }
  L.slab = p;
  p = sh_align(p + slab_bytes);
  L.end = p;
  return L;
}
// meta row of one (source, destination) pair: rows per level, then slab bytes per level
inline u64 blob_bytes(const u64 *meta) {
  u64 p = 0;
  for (int l = 0; l < L_NLEVELS; l++) p = level_layout(l, p, meta[l], meta[L_NLEVELS + l]).end;
  return p;
}

// ------------------------------------------------------------------ device-side descriptors

struct LevelSrc {  // where a level's rows come from (device pointers)
  const gar_str *str[SH_MAX_STR];
  const u8 *u8c[SH_MAX_U8];
  const u32 *u32c[SH_MAX_U32];
  const u32 *gid;  // explicit global ids (rows that already travelled once), else gid_base + row
  u32 gid_base;
  const u32 *child_begin[SH_MAX_CHILD];
  const u8 *child_dest[SH_MAX_CHILD];  // nullable: child c follows its parent only to destination child_dest[c]
  const u8 *slab;
  u32 n;
};
struct LevelPlan {  // selection of one level: rows sel[0..*m) sorted by destination
  u32 *sel;
  u32 *m;         // device scalar
  u32 cap;        // host upper bound of *m
  u32 *row_off;   // device [n_ranks+1]
  u32 *slab_scan; // [cap+1] exclusive scan of the rows' string bytes
  u32 *slab_off;  // device [n_ranks+1]
  u32 *cnt[SH_MAX_CHILD];  // [cap+1] exclusive scan of child counts per link
  u32 multi;      // host-side note: a source row may be selected for several destinations (children can outnumber the source level)
};

// strings start 8-byte aligned inside a blob: the copy is whole words (unaligned 8-byte loads, aligned stores)
GAR_HD u32 sh_pad8(u32 len) { return (len + 7u) & ~7u; }
GAR_HD u32 shard_of(u64 h, u32 n_ranks) { return (u32)(xx_avalanche(h + 0x9E3779B97F4A7C15ull) >> 33) % n_ranks; }
// The key of the two by-hostname lookups (GetLoadBalancer by (region, name) of the tokenised hostname, global_accelerator.go:116-120;
// ListGlobalAcceleratorByHostname by the hostname itself, :62-85): one function of the hostname string, so the probe, the
// LB it resolves to and every accelerator tagged with that hostname meet on one shard.
GAR_HD u64 directory_key(u8 code, Str host, Str region, Str name) { return code <= GAR_TOK_NLB ? key_hash_lb(region, name) : gar_hash(host); }
GAR_HD u32 dest_of(u32 j, const u32 *row_off, u32 n_ranks) {
  u32 d = 0;
  while (d + 1 < n_ranks && j >= row_off[d + 1]) d++;
  return d;
}

// ------------------------------------------------------------------ routing keys (round 1)

struct FShKeyObj {
  Work W;
  u32 G;
  u32 *keys, *vals;
  GAR_HD void operator()(u32 i) const {
    keys[i] = shard_of(W.okey_hash[i], G);
    vals[i] = i;
  }
};
struct FShObjKey {  // the "ns/name" key as one string + where it splits
  DevTables T;
  gar_str *key;
  u32 *ns_len;
  GAR_HD void operator()(u32 i) const {
    gar_str ns = T.o.obj_ns[i];
    key[i] = GAR_STR(GAR_STR_OFF(ns), GAR_STR_LEN(ns) + 1 + GAR_STR_LEN(T.o.obj_name[i]));
    ns_len[i] = (u32)GAR_STR_LEN(ns);
  }
};
struct FShKeyLb {
  DevTables T;
  u32 G;
  u32 *keys, *vals;
  GAR_HD void operator()(u32 i) const {
    keys[i] = shard_of(key_hash_lb(mkstr(T.a.slab, T.a.lb_region[i]), mkstr(T.a.slab, T.a.lb_name[i])), G);
    vals[i] = i;
  }
};
struct FShKeyAcc {  // own rows: what ListGlobalAcceleratorByResource can return and what the orphan pass inspects
  Work W;
  u32 G;
  u32 *keys, *vals;
  GAR_HD void operator()(u32 a) const {
    u32 fl = W.acc_flags[a];
    keys[a] = ((fl & ACC_MINE) && (fl & ACC_OWNER_KEYED)) ? shard_of(W.acc_owner_hash[a], G) : SH_DROP;
    vals[a] = a;
  }
};
struct FShKeyStub {  // what ListGlobalAcceleratorByHostname can return
  DevTables T;
  Work W;
  u32 G;
  u32 *keys, *vals;
  GAR_HD void operator()(u32 a) const {
    u32 k = SH_DROP;
    if (W.acc_flags[a] & ACC_MINE) {
      gar_str th = W.acc_thost[a], name, region;
      Str h = mkstr(T.a.slab, th);
      u8 code = tokenise_str(h, GAR_STR_OFF(th), &name, &region);
      k = shard_of(directory_key(code, h, mkstr(T.a.slab, region), mkstr(T.a.slab, name)), G);
    }
    keys[a] = k;
    vals[a] = a;
  }
};
struct FShKeyProbe {
  DevTables T;
  Work W;
  const u32 *lbi_obj;
  u32 G;
  u32 *keys, *vals, *home;
  GAR_HD void operator()(u32 l) const {
    Str h = mkstr(T.o.slab, T.o.lbi_hostname[l]);
    keys[l] = shard_of(directory_key(W.tok_code[l], h, mkstr(T.o.slab, W.tok_region[l]), mkstr(T.o.slab, W.tok_name[l])), G);
    vals[l] = l;
    home[l] = shard_of(W.okey_hash[lbi_obj[l]], G);
  }
};
// a stub only answers ListGlobalAcceleratorByHostname: of its tags only the three that lookup reads travel with it
struct FShStubTagKeep {
  DevTables T;
  u8 *keep;
  GAR_HD void operator()(u32 t) const {
    Str k = mkstr(T.a.slab, T.a.tag_key[t]);
    keep[t] = (STREQ_LIT(k, TAG_MANAGED) || STREQ_LIT(k, TAG_THOST) || STREQ_LIT(k, TAG_CLUSTER)) ? (u8)SH_FOLLOW : (u8)SH_DROP;
  }
};
struct FShValDest {
  Work W;
  u32 G;
  u8 *val_dest;
  GAR_HD void operator()(u32 v) const { val_dest[v] = W.val_cls[v] == VAL_NOT_OWNER ? (u8)SH_DROP : (u8)shard_of(W.val_key_hash[v], G); }
};
// Which shards need a record: bit d of mask[rec] for the record of every owner value homed on d, and for every alias record
// under the same (zone, name) (FindOwneredARecordSets, route53.go:216-238).
struct FShRecMask {
  DevTables T;
  Work W;
  const u8 *val_dest;
  u32 *mask;  // [n_records]
  GAR_HD void operator()(u32 v) const {
    u32 d = val_dest[v];
    if (d == SH_DROP) return;
    u32 rec = W.val_rec[v], zone = W.rec_zone[rec];
    const u32 bit = 1u << d;
    if (!(mask[rec] & bit)) GAR_ATOMIC_OR(&mask[rec], bit);
    Str name = mkstr(T.a.slab, T.a.rec_name[rec]);
    Cursor c = idx_open(W.ix_alias, key_hash_zoned_h(zone, W.rec_name_hash[rec]));
    IdxEntry e;
    while (idx_next(W.ix_alias, c, &e)) {
      if (e.a0 != zone || e.row == rec || !streq(mkstr(T.a.slab, e.s0), name)) continue;
      if (!(mask[e.row] & bit)) GAR_ATOMIC_OR(&mask[e.row], bit);
    }
  }
};
struct FShIota {
  u32 *keys, *vals;
  u32 key;
  GAR_HD void operator()(u32 i) const {
    keys[i] = key;
    vals[i] = i;
  }
};

// ------------------------------------------------------------------ selection lists

// keys sorted ascending; row_off[d] = first position with key >= d (d = 0..G); *m = row_off[G]
struct FShSelBounds {
  const u32 *keys;
  u32 n, G;
  u32 *row_off, *m;
  GAR_HD void operator()(u32 d) const {
    u32 lo = 0, hi = n;
    while (lo < hi) {
      u32 mid = (lo + hi) >> 1;
      if (keys[mid] < d) lo = mid + 1;
      else hi = mid;
    }
    row_off[d] = lo;
    if (d == G) *m = lo;
  }
};
// Destination masks -> the selection list sorted by (destination, row), duplicates impossible.  One thread per tile of 32 rows:
// count per destination, one scan over the [destination][tile] counts, then the same threads write their rows.
constexpr u32 SH_MASK_TILE = 32;
struct FShMaskCount {
  const u32 *mask;
  u32 n, G, T;
  u32 *counts;  // [G * T + 1], destination-major
  GAR_HD void operator()(u32 t) const {
    u32 c[SH_MAX_RANKS];
    for (int d = 0; d < SH_MAX_RANKS; d++) c[d] = 0;
    u32 r1 = (t + 1) * SH_MASK_TILE < n ? (t + 1) * SH_MASK_TILE : n;
    for (u32 r = t * SH_MASK_TILE; r < r1; r++) {
      u32 m = mask[r];
      for (int d = 0; d < SH_MAX_RANKS; d++) c[d] += (m >> d) & 1u;
    }
    for (int d = 0; d < SH_MAX_RANKS; d++)
      if ((u32)d < G) counts[(size_t)d * T + t] = c[d];
  }
};
struct FShMaskFill {
  const u32 *mask;
  u32 n, G, T;
  const u32 *scanned;
  u32 *sel;
  GAR_HD void operator()(u32 t) const {
    u32 pos[SH_MAX_RANKS];
    for (int d = 0; d < SH_MAX_RANKS; d++) pos[d] = (u32)d < G ? scanned[(size_t)d * T + t] : 0;
    u32 r1 = (t + 1) * SH_MASK_TILE < n ? (t + 1) * SH_MASK_TILE : n;
    for (u32 r = t * SH_MASK_TILE; r < r1; r++) {
      u32 m = mask[r];
      for (int d = 0; d < SH_MAX_RANKS; d++)
        if ((m >> d) & 1u) sel[pos[d]++] = r;
    }
  }
};
struct FShMaskBounds {
  const u32 *scanned;
  u32 G, T;
  u32 *row_off, *m;
  GAR_HD void operator()(u32 d) const {
    u32 v = scanned[(size_t)d * T];
    row_off[d] = v;
    if (d == G) *m = v;
  }
};
struct FShChildFill {
  LevelSrc src;
  int link;
  LevelPlan P;
  u32 G;
  u32 *child_sel;
  GAR_HD void operator()(u32 j) const {
    if (j >= *P.m) return;
    u32 p = P.sel[j], b0 = src.child_begin[link][p], b1 = src.child_begin[link][p + 1];
    u32 pos = P.cnt[link][j];
    const u8 *cd = src.child_dest[link];
    if (cd) {
      u32 d = dest_of(j, P.row_off, G);
      for (u32 ch = b0; ch < b1; ch++)
        if (cd[ch] == d || cd[ch] == SH_FOLLOW) child_sel[pos++] = ch;
    } else {
      for (u32 ch = b0; ch < b1; ch++) child_sel[pos++] = ch;
    }
  }
};
// boundaries of a derived list (children, string bytes): value of the parent's scan at the parent's boundaries
struct FShDerivedBounds {
  const u32 *parent_row_off, *scanned;
  u32 G;
  u32 *out_off, *out_m;
  GAR_HD void operator()(u32 d) const {
    u32 v = scanned[parent_row_off[d]];
    out_off[d] = v;
    if (d == G && out_m) *out_m = v;
  }
};
// child counts of every link and the string bytes of a selected row, one pass over the selection
struct FShRowSizes {
  LevelSrc src;
  LevelSchema S;
  LevelPlan P;
  u32 G;
  GAR_HD void operator()(u32 j) const {
    u32 cnt[SH_MAX_CHILD] = {0, 0, 0}, bytes = 0;
    if (j < *P.m) {
      u32 p = P.sel[j], d = 0;
      bool need_d = false;
      for (int c = 0; c < SH_MAX_CHILD; c++) need_d |= c < S.n_child && src.child_dest[c] != nullptr;
      if (need_d) d = dest_of(j, P.row_off, G);
      for (int c = 0; c < SH_MAX_CHILD; c++) {
        if (c >= S.n_child) break;
        u32 b0 = src.child_begin[c][p], b1 = src.child_begin[c][p + 1];
        const u8 *cd = src.child_dest[c];
        if (cd) {
          for (u32 ch = b0; ch < b1; ch++) cnt[c] += cd[ch] == d || cd[ch] == SH_FOLLOW;
        } else {
          cnt[c] = b1 - b0;
        }
      }
      for (int c = 0; c < SH_MAX_STR; c++)
        if (c < S.n_str) bytes += sh_pad8((u32)GAR_STR_LEN(src.str[c][p]));
    }
    for (int c = 0; c < SH_MAX_CHILD; c++)
      if (c < S.n_child) P.cnt[c][j] = cnt[c];
    P.slab_scan[j] = bytes;
  }
};

// ------------------------------------------------------------------ pack

struct PackDst {
  u8 *base[SH_MAX_RANKS];  // start of destination d's blob
  LevelLayout lay[SH_MAX_RANKS];
};
// One thread per selected row: its fixed-width columns, then its strings, each copied as whole 8-byte words (the source may sit
// at any byte offset: aligned loads + funnel shift, one load per word; the destination word is aligned; the bytes behind a
// string's end up to the next word are don't-care).  A row's strings are ~30-250 bytes, so a thread keeps that many bytes in
// flight behind ONE dependent chain (selection -> string refs -> bytes) — the 8-lanes-per-row version of round 1 moved 8 bytes
// per chain and ran at 1.4 TB/s.  Strings longer than SH_LONG_WORDS words are cut here and finished by FShPackLong.
constexpr u32 SH_LONG_WORDS = 256;  // 2 KB
GAR_HD void sh_copy_words(u64 *dst, const u8 *s, u32 words) {
  if (!words) return;
  uintptr_t a = (uintptr_t)s;
  const u64 *q = (const u64 *)(a & ~(uintptr_t)7);
  const unsigned sh = (unsigned)(a & 7) * 8;
  u64 lo = q[0];
#pragma unroll 4
  for (u32 w = 0; w < words; w++) {
    u64 hi = q[w + 1];
    dst[w] = (lo >> sh) | ((hi << 1) << (63 - sh));
    lo = hi;
  }
}
struct FShPackRows {
  LevelSrc src;
  LevelSchema S;
  LevelPlan P;
  u32 G;
  PackDst D;
  u32 *any_long;  // device flag: some string was cut
  // straight to the destination, long strings cut (FShPackLong copies the rest)
  GAR_HD void operator()(u32 j) const {
    u32 d = dest_of(j, P.row_off, G), k = j - P.row_off[d], p = P.sel[j];
    u8 *b = D.base[d];
    const LevelLayout &L = D.lay[d];
    u64 off = P.slab_scan[j] - P.slab_scan[P.row_off[d]];
    gar_str ref[SH_MAX_STR];
    for (int c = 0; c < SH_MAX_STR; c++)
      if (c < S.n_str) ref[c] = src.str[c][p];
    for (int c = 0; c < S.n_u8; c++) (b + L.u8c[c])[k] = src.u8c[c][p];
    for (int c = 0; c < S.n_u32; c++) ((u32 *)(b + L.u32c[c]))[k] = src.u32c[c][p];
    if (S.has_gid) ((u32 *)(b + L.gid))[k] = src.gid ? src.gid[p] : src.gid_base + p;
    for (int c = 0; c < S.n_child; c++) ((u32 *)(b + L.cnt[c]))[k] = P.cnt[c][j + 1] - P.cnt[c][j];
    bool cut = false;
    for (int c = 0; c < SH_MAX_STR; c++) {
      if (c >= S.n_str) break;
      u64 len = GAR_STR_LEN(ref[c]);
      ((gar_str *)(b + L.str[c]))[k] = GAR_STR(off, len);
      u32 words = sh_pad8((u32)len) >> 3;
      cut |= words > SH_LONG_WORDS;
      sh_copy_words((u64 *)(b + L.slab + off), src.slab + GAR_STR_OFF(ref[c]), words > SH_LONG_WORDS ? SH_LONG_WORDS : words);
      off += (u64)words << 3;
    }
    if (cut) *any_long = 1;
  }
};
// The rest of the cut strings: a fixed number of workers stride over the rows, SH_COPY_LANES lanes per row.  Leaves at once when
// no string was cut (the flag stays on the device: no host round-trip decides about this launch).
constexpr u32 SH_COPY_LANES = 8, SH_LONG_WORKERS = 148 * 8 * 256;
struct FShPackLong {
  LevelSrc src;
  int n_str;
  LevelPlan P;
  u32 G, m;
  PackDst D;
  const u32 *any_long;
  GAR_HD void operator()(u32 t) const {
    if (!*any_long) return;
    const u32 lane = t % SH_COPY_LANES;
    for (u32 j = t / SH_COPY_LANES; j < m; j += SH_LONG_WORKERS / SH_COPY_LANES) {
      u32 d = dest_of(j, P.row_off, G), p = P.sel[j];
      u64 *dst = (u64 *)(D.base[d] + D.lay[d].slab + (P.slab_scan[j] - P.slab_scan[P.row_off[d]]));
      for (int c = 0; c < n_str; c++) {
        gar_str r = src.str[c][p];
        const u8 *s = src.slab + GAR_STR_OFF(r);
        u32 words = sh_pad8((u32)GAR_STR_LEN(r)) >> 3;
        for (u32 w = SH_LONG_WORDS + lane; w < words; w += SH_COPY_LANES) dst[w] = ld64u(s + 8 * (size_t)w);
        dst += words;
      }
    }
  }
};

// ------------------------------------------------------------------ unpack (merge the received blobs of one level)

struct SegSrc {
  const u8 *base;
  LevelLayout lay;
};
struct UnpackDst {
  gar_str *str[SH_MAX_STR];
  u8 *u8c[SH_MAX_U8];
  u32 *u32c[SH_MAX_U32];
  u32 *gid;
  u32 *cnt[SH_MAX_CHILD];  // raw child counts (the caller scans them into CSR begins); nullable
};
struct FShUnpackCols {
  int nseg;
  SegSrc seg[SH_MAX_SEGS];
  u8 has_cnt[SH_MAX_SEGS][SH_MAX_CHILD];  // a segment of a level without that child link (stubs have no listeners) reads as 0
  u32 seg_row[SH_MAX_SEGS + 1];
  u64 slab_base[SH_MAX_SEGS];  // where segment s's string bytes start in the merged slab
  LevelSchema S;
  UnpackDst D;
  GAR_HD void operator()(u32 j) const {
    int s = 0;
    while (s + 1 < nseg && j >= seg_row[s + 1]) s++;
    u32 k = j - seg_row[s];
    const u8 *b = seg[s].base;
    const LevelLayout &L = seg[s].lay;
    for (int c = 0; c < S.n_str; c++) {
      gar_str r = ((const gar_str *)(b + L.str[c]))[k];
      D.str[c][j] = GAR_STR(GAR_STR_OFF(r) + slab_base[s], GAR_STR_LEN(r));
    }
    for (int c = 0; c < S.n_u8; c++) D.u8c[c][j] = (b + L.u8c[c])[k];
    for (int c = 0; c < S.n_u32; c++) D.u32c[c][j] = ((const u32 *)(b + L.u32c[c]))[k];
    if (S.has_gid) D.gid[j] = ((const u32 *)(b + L.gid))[k];
    for (int c = 0; c < S.n_child; c++)
      if (D.cnt[c]) D.cnt[c][j] = has_cnt[s][c] ? ((const u32 *)(b + L.cnt[c]))[k] : 0u;
  }
};
struct FShObjNsName {
  const gar_str *key;
  const u32 *ns_len;
  gar_str *ns, *name;
  GAR_HD void operator()(u32 i) const {
    u64 off = GAR_STR_OFF(key[i]), len = GAR_STR_LEN(key[i]), nl = ns_len[i];
    ns[i] = GAR_STR(off, nl);
    name[i] = GAR_STR(off + nl + 1, len - nl - 1);
  }
};
// records arrive zone-major (whole zones per source rank, zone ranges ascending with the rank): begin[z] = first record
// whose zone is >= z
struct FShZoneBegin {
  const u32 *rec_zone;
  u32 n_rec;
  u32 *begin;
  GAR_HD void operator()(u32 z) const {
    u32 lo = 0, hi = n_rec;
    while (lo < hi) {
      u32 mid = (lo + hi) >> 1;
      if (rec_zone[mid] < z) lo = mid + 1;
      else hi = mid;
    }
    begin[z] = lo;
  }
};

// sharded-mode contract checks: the zone table must be the same on every rank (fingerprint travels in the meta row), and the
// merged record sets must come out zone-major
struct FShZoneFingerprint {
  DevTables T;
  unsigned long long *acc;
  GAR_HD void operator()(u32 z) const {
    u64 h = hmix((u64)z + 1, gar_hash(mkstr(T.a.slab, T.a.zone_name[z])));
#if defined(__CUDA_ARCH__)
    atomicAdd(acc, (unsigned long long)h);
#else
    *acc += h;
#endif
  }
};
struct FShCheckZoneOrder {
  const u32 *rec_zone;
  u32 n_zones;
  u32 *bad;
  GAR_HD void operator()(u32 r) const {
    if (rec_zone[r] >= n_zones || (r > 0 && rec_zone[r - 1] > rec_zone[r])) GAR_ATOMIC_ADD(bad, 1u);
  }
};
constexpr int SH_META_ZONE_FP = 2 * L_NLEVELS;  // meta word carrying the sender's zone-table fingerprint
#define GAR_E_SHARD_CONTRACT 2000               // Sharder: the slices violate the sharded-mode contract (mapped to GAR_E_INVALID)

// ------------------------------------------------------------------ directory: answer the probes (round 2 selection)

// One probe = one lbIngress hostname of some object.  The LB the reference would get (first row wins) and the first two
// accelerators ListGlobalAcceleratorByHostname would return go to the probe's home shard.
struct FShAnswer {
  DevTables T;  // directory tables: lbi_* = probes, lb_* and acc_* = rows routed here
  Work W;
  const u32 *home;
  u32 *lb_mask, *stub_mask;  // [n_lbs], [n_accels]: bit d = the row is an answer for a probe whose object lives on shard d
  GAR_HD void operator()(u32 p) const {
    const u32 bit = 1u << home[p];
    if (W.tok_code[p] <= GAR_TOK_NLB) {
      u32 st;
      u32 lb = find_lb(T, W, mkstr(T.o.slab, W.tok_region[p]), mkstr(T.o.slab, W.tok_name[p]), &st);
      if (lb != GAR_NONE && !(lb_mask[lb] & bit)) GAR_ATOMIC_OR(&lb_mask[lb], bit);
    }
    Str host = mkstr(T.o.slab, T.o.lbi_hostname[p]);
    Cursor c = idx_open(W.ix_thost, key_hash_str(host));
    IdxEntry e;
    u32 k = 0;
    while (k < 2 && idx_next(W.ix_thost, c, &e)) {
      if (!streq(mkstr(T.a.slab, e.s0), host)) continue;
      if (!(stub_mask[e.row] & bit)) GAR_ATOMIC_OR(&stub_mask[e.row], bit);
      k++;
    }
  }
};

// ------------------------------------------------------------------ results: local rows -> global ids

struct ShGids {
  const u32 *obj, *lb, *acc, *lis, *eg, *rec, *val;
};
struct FShTranslateOps {
  gar_op *ops;
  ShGids g;
  GAR_HD u32 m(const u32 *tab, u32 v) const { return v >= GAR_PENDING ? v : tab[v]; }  // GAR_NONE / GAR_PENDING name no row
  GAR_HD void operator()(u32 k) const {
    gar_op o = ops[k];
    o.obj = m(g.obj, o.obj);
    switch (o.head & 0xFFu) {
      case GAR_OP_GA_CREATE_CHAIN: o.a0 = m(g.lb, o.a0); break;
      case GAR_OP_GA_UPDATE_ACCEL: o.a0 = m(g.acc, o.a0); o.a1 = m(g.lb, o.a1); break;
      case GAR_OP_GA_CREATE_LISTENER: o.a0 = m(g.acc, o.a0); break;
      case GAR_OP_GA_UPDATE_LISTENER: o.a0 = m(g.acc, o.a0); o.a1 = m(g.lis, o.a1); break;
      case GAR_OP_GA_CREATE_EG: o.a0 = m(g.acc, o.a0); o.a1 = m(g.lis, o.a1); o.a2 = m(g.lb, o.a2); break;
      case GAR_OP_GA_UPDATE_EG: o.a0 = m(g.acc, o.a0); o.a1 = m(g.eg, o.a1); o.a2 = m(g.lb, o.a2); break;
      case GAR_OP_GA_DELETE_CHAIN: o.a0 = m(g.acc, o.a0); o.a1 = m(g.lis, o.a1); o.a2 = m(g.eg, o.a2); break;
      case GAR_OP_R53_CREATE: o.a1 = m(g.acc, o.a1); break;  // a0 = zone: the zone table is the same on every rank
      case GAR_OP_R53_UPSERT_A: o.a1 = m(g.acc, o.a1); o.a2 = m(g.rec, o.a2); break;
      case GAR_OP_R53_DELETE_RECORD: o.a1 = m(g.rec, o.a1); o.a2 = m(g.val, o.a2); break;
      default: break;
    }
    ops[k] = o;
  }
};

// ------------------------------------------------------------------ host-side driver

template <class B>
struct Sharder {
  B &be;
  gar_shard cfg{};
  u32 G = 1;
  DevTables S{};                     // this rank's slice
  Pipeline<B> *slice_pipe = nullptr; // row-local pass over the slice
  Pipeline<B> *dir_pipe = nullptr;   // directory tables + their indexes
  DevTables Dt{};                    // directory tables
  const u32 *dir_home = nullptr, *dir_lb_gid = nullptr, *dir_stub_gid = nullptr;
  DevTables H{};                     // home sub-snapshot (result)
  ShGids gids{};
  u32 guest_from = 0;

  // current plan
  LevelSrc src[L_NLEVELS]{};
  LevelPlan plan[L_NLEVELS]{};
  bool active[L_NLEVELS]{};
  u32 *bounds_dev = nullptr;  // [L_NLEVELS][2][SH_MAX_RANKS+1]
  u32 h_row_off[L_NLEVELS][SH_MAX_RANKS + 1]{}, h_slab_off[L_NLEVELS][SH_MAX_RANKS + 1]{};
  // round 1 receive side, kept for the home merge after round 2
  const u8 *recv1 = nullptr;
  u64 meta1[SH_MAX_RANKS][GAR_SHARD_META_WORDS]{};
  u64 zone_fp = 0;           // fingerprint of this rank's zone table (round 1 meta)
  const char *contract_error = nullptr;

  bool copy_merge = false;   // GAR_SHARD_COPY_MERGE=1: always copy the received string bytes into merged slabs (A/B, tests)

  explicit Sharder(B &b) : be(b) {
    const char *cm = getenv("GAR_SHARD_COPY_MERGE");
    copy_merge = cm && cm[0] == '1';
  }
  ~Sharder() {
    delete slice_pipe;
    delete dir_pipe;
  }

  template <class Tp>
  Tp *alloc(int arena, size_t count) { return (Tp *)be.shard_alloc(arena, sizeof(Tp) * (count + 1)); }
  u32 *row_off_dev(int l) { return bounds_dev + (size_t)l * 2 * (SH_MAX_RANKS + 1); }
  u32 *slab_off_dev(int l) { return row_off_dev(l) + (SH_MAX_RANKS + 1); }

  void plan_begin() {
    be.shard_reset(SH_ARENA_PLAN);
    bounds_dev = alloc<u32>(SH_ARENA_PLAN, (size_t)L_NLEVELS * 2 * (SH_MAX_RANKS + 1) + 2 * L_NLEVELS);
    be.fill32(bounds_dev, 0, (size_t)L_NLEVELS * 2 * (SH_MAX_RANKS + 1) + 2 * L_NLEVELS);
    for (int l = 0; l < L_NLEVELS; l++) {
      active[l] = false;
      src[l] = LevelSrc{};
      plan[l] = LevelPlan{};
    }
  }
  u32 *m_dev(int l) { return bounds_dev + (size_t)L_NLEVELS * 2 * (SH_MAX_RANKS + 1) + l; }

  // top-level selection from (keys, vals) that are already in their final (key, val) order; keys >= G are dropped
  void set_top(int l, u32 *keys, u32 *vals, u32 n, bool multi = false) {
    active[l] = true;
    plan[l].multi = multi;
    plan[l].sel = vals;
    plan[l].cap = n;
    plan[l].m = m_dev(l);
    plan[l].row_off = row_off_dev(l);
    plan[l].slab_off = slab_off_dev(l);
    be.for_each("shard_bounds", G + 1, FShSelBounds{keys, n, G, plan[l].row_off, plan[l].m});
  }
  // single-destination level: one key per source row, stable partition by destination
  template <class KeyF>
  void top_single(int l, u32 n, KeyF make) {
    u32 *keys = alloc<u32>(SH_ARENA_PLAN, n), *vals = alloc<u32>(SH_ARENA_PLAN, n);
    u32 *k2 = alloc<u32>(SH_ARENA_PLAN, n), *v2 = alloc<u32>(SH_ARENA_PLAN, n);
    if (n) {
      be.for_each("shard_keys", n, make(keys, vals));
      be.sort_pairs(keys, vals, k2, v2, n, 8);
    }
    set_top(l, keys, vals, n);
  }
  // children of level l (whose plan is set), then its string bytes
  void plan_children_and_strings(int l) {
    const LevelSchema &Sc = SH_SCHEMA[l];
    LevelPlan &P = plan[l];
    for (int c = 0; c < Sc.n_child; c++) P.cnt[c] = alloc<u32>(SH_ARENA_PLAN, (size_t)P.cap + 1);
    P.slab_scan = alloc<u32>(SH_ARENA_PLAN, (size_t)P.cap + 1);
    be.for_each("shard_row_sizes", P.cap + 1, FShRowSizes{src[l], Sc, P, G});
    for (int c = 0; c < Sc.n_child; c++) {
      int ch = Sc.child[c];
      be.exclusive_scan(P.cnt[c], P.cap + 1);
      active[ch] = true;
      plan[ch].cap = src[ch].n;
      plan[ch].multi = P.multi;
      if (P.multi && !src[l].child_dest[c]) be.download(&plan[ch].cap, P.cnt[c] + P.cap, 4);  // replicated parents: exact child count
      plan[ch].sel = alloc<u32>(SH_ARENA_PLAN, plan[ch].cap);
      plan[ch].m = m_dev(ch);
      plan[ch].row_off = row_off_dev(ch);
      plan[ch].slab_off = slab_off_dev(ch);
      if (P.cap) be.for_each("shard_child_fill", P.cap, FShChildFill{src[l], c, P, G, plan[ch].sel});
      be.for_each("shard_child_bounds", G + 1, FShDerivedBounds{P.row_off, P.cnt[c], G, plan[ch].row_off, plan[ch].m});
    }
    if (Sc.n_str) be.exclusive_scan(P.slab_scan, P.cap + 1);
    be.for_each("shard_slab_bounds", G + 1, FShDerivedBounds{P.row_off, P.slab_scan, G, P.slab_off, nullptr});
  }
  // after every level is planned: bring the boundaries to the host and fill the meta rows
  void plan_finish(u64 *meta /* [G][GAR_SHARD_META_WORDS] */, u64 *send_bytes) {
    for (int l = 0; l < L_NLEVELS; l++)
      if (active[l]) plan_children_and_strings(l);  // parents precede their children in ShLevel order
    std::vector<u32> h((size_t)L_NLEVELS * 2 * (SH_MAX_RANKS + 1));
    be.download(h.data(), bounds_dev, 4 * h.size());
    for (int l = 0; l < L_NLEVELS; l++)
      for (u32 d = 0; d <= G; d++) {
        h_row_off[l][d] = active[l] ? h[((size_t)l * 2) * (SH_MAX_RANKS + 1) + d] : 0;
        h_slab_off[l][d] = active[l] ? h[((size_t)l * 2 + 1) * (SH_MAX_RANKS + 1) + d] : 0;
      }
    for (u32 d = 0; d < G; d++) {
      u64 *row = meta + (size_t)d * GAR_SHARD_META_WORDS;
      for (int w = 0; w < GAR_SHARD_META_WORDS; w++) row[w] = 0;
      for (int l = 0; l < L_NLEVELS; l++) {
        row[l] = h_row_off[l][d + 1] - h_row_off[l][d];
        row[L_NLEVELS + l] = h_slab_off[l][d + 1] - h_slab_off[l][d];
      }
      row[SH_META_ZONE_FP] = zone_fp;  // not part of the layout: blob_bytes ignores it
      send_bytes[d] = blob_bytes(row);
    }
  }

  // ---- round 1: route the slice
  void route1(const DevTables &slice, const gar_shard &c, u64 *meta, u64 *send_bytes) {
    cfg = c;
    G = c.n_ranks;
    S = slice;
    delete slice_pipe;
    slice_pipe = new Pipeline<B>(be, S);
    slice_pipe->prepare_route();
    const Work &W = slice_pipe->W;
    const gar_objects &O = S.o;
    const gar_actual &A = S.a;
    plan_begin();
    {
      unsigned long long *fp = (unsigned long long *)alloc<u64>(SH_ARENA_PLAN, 2);
      be.fill32((u32 *)fp, 0, 4);
      if (A.n_zones) be.for_each("shard_zone_fingerprint", A.n_zones, FShZoneFingerprint{S, fp});
      be.download(&zone_fp, fp, 8);
      zone_fp ^= (u64)A.n_zones << 48;
    }
    // sources
    gar_str *okey = alloc<gar_str>(SH_ARENA_PLAN, O.n_objects);
    u32 *ns_len = alloc<u32>(SH_ARENA_PLAN, O.n_objects);
    if (O.n_objects) be.for_each("shard_obj_key", O.n_objects, FShObjKey{S, okey, ns_len});
    u32 *lbi_obj = alloc<u32>(SH_ARENA_PLAN, O.n_lbi);
    if (O.n_lbi) be.for_each("expand_lbi_obj", O.n_lbi, FExpand{O.obj_lbi_begin, O.n_objects, lbi_obj});
    u32 *probe_home = alloc<u32>(SH_ARENA_PLAN, O.n_lbi);
    u8 *val_dest = alloc<u8>(SH_ARENA_PLAN, A.n_values);
    if (A.n_values) be.for_each("shard_val_dest", A.n_values, FShValDest{W, G, val_dest});

    LevelSrc x{};
    x = LevelSrc{}; x.str[0] = okey; x.str[1] = O.obj_ingress_class; x.u8c[0] = O.obj_kind; x.u8c[1] = O.obj_spec_type; x.u8c[2] = O.obj_flags;
    x.u32c[0] = ns_len; x.gid_base = c.obj_base; x.child_begin[0] = O.obj_ann_begin; x.child_begin[1] = O.obj_lbi_begin; x.child_begin[2] = O.obj_port_begin;
    x.slab = O.slab; x.n = O.n_objects; src[L_OBJ] = x;
    x = LevelSrc{}; x.str[0] = O.ann_key; x.str[1] = O.ann_val; x.slab = O.slab; x.n = O.n_ann; src[L_ANN] = x;
    x = LevelSrc{}; x.str[0] = O.lbi_hostname; x.slab = O.slab; x.n = O.n_lbi; src[L_LBI] = x;
    x = LevelSrc{}; x.str[0] = O.port_proto; x.u32c[0] = (const u32 *)O.port_number; x.slab = O.slab; x.n = O.n_ports; src[L_PORT] = x;
    x = LevelSrc{}; x.str[0] = A.acc_name; x.str[1] = A.acc_dns; x.u8c[0] = A.acc_enabled; x.gid_base = c.acc_base;
    x.child_begin[0] = A.acc_tag_begin; x.child_begin[1] = A.acc_lis_begin; x.slab = A.slab; x.n = A.n_accels; src[L_ACC] = x;
    x.child_begin[1] = nullptr;
    u8 *stub_tag_keep = alloc<u8>(SH_ARENA_PLAN, A.n_tags);
    if (A.n_tags) be.for_each("shard_stub_tag_keep", A.n_tags, FShStubTagKeep{S, stub_tag_keep});
    x.child_dest[0] = stub_tag_keep;
    src[L_STUB] = x;
    x = LevelSrc{}; x.str[0] = A.tag_key; x.str[1] = A.tag_val; x.slab = A.slab; x.n = A.n_tags; src[L_TAG] = x; src[L_STUBTAG] = x;
    x = LevelSrc{}; x.u8c[0] = A.lis_proto; x.gid_base = c.lis_base; x.child_begin[0] = A.lis_pr_begin; x.child_begin[1] = A.lis_eg_begin;
    x.slab = A.slab; x.n = A.n_listeners; src[L_LIS] = x;
    x = LevelSrc{}; x.u32c[0] = (const u32 *)A.pr_from; x.slab = A.slab; x.n = A.n_port_ranges; src[L_PR] = x;
    x = LevelSrc{}; x.gid_base = c.eg_base; x.child_begin[0] = A.eg_ep_begin; x.slab = A.slab; x.n = A.n_egs; src[L_EG] = x;
    x = LevelSrc{}; x.str[0] = A.ep_id; x.slab = A.slab; x.n = A.n_endpoints; src[L_EP] = x;
    x = LevelSrc{}; x.str[0] = A.rec_name; x.str[1] = A.rec_alias_dns; x.u8c[0] = A.rec_type; x.u8c[1] = A.rec_has_alias; x.u32c[0] = W.rec_zone;
    x.gid_base = c.rec_base; x.child_begin[0] = A.rec_val_begin; x.child_dest[0] = val_dest; x.slab = A.slab; x.n = A.n_records; src[L_REC] = x;
    x = LevelSrc{}; x.str[0] = A.val_value; x.gid_base = c.val_base; x.slab = A.slab; x.n = A.n_values; src[L_VAL] = x;
    x = LevelSrc{}; x.str[0] = A.zone_name; x.slab = A.slab; x.n = A.n_zones; src[L_ZONE] = x;
    x = LevelSrc{}; x.str[0] = A.lb_region; x.str[1] = A.lb_name; x.str[2] = A.lb_dns; x.str[3] = A.lb_arn; x.u8c[0] = A.lb_state; x.gid_base = c.lb_base;
    x.slab = A.slab; x.n = A.n_lbs; src[L_LB] = x;
    x = LevelSrc{}; x.str[0] = O.lbi_hostname; x.u32c[0] = probe_home; x.slab = O.slab; x.n = O.n_lbi; src[L_PROBE] = x;

    // top-level selections
    const DevTables Sl = S;
    const u32 Gn = G;
    top_single(L_OBJ, O.n_objects, [&](u32 *k, u32 *v) { return FShKeyObj{W, Gn, k, v}; });
    top_single(L_ACC, A.n_accels, [&](u32 *k, u32 *v) { return FShKeyAcc{W, Gn, k, v}; });
    top_single(L_LB, A.n_lbs, [&](u32 *k, u32 *v) { return FShKeyLb{Sl, Gn, k, v}; });
    top_single(L_STUB, A.n_accels, [&](u32 *k, u32 *v) { return FShKeyStub{Sl, W, Gn, k, v}; });
    top_single(L_PROBE, O.n_lbi, [&](u32 *k, u32 *v) { return FShKeyProbe{Sl, W, lbi_obj, Gn, k, v, probe_home}; });
    {  // the zone table stays where it is: every rank already holds all of it (sharded-mode contract)
      u32 nz = A.n_zones;
      u32 *keys = alloc<u32>(SH_ARENA_PLAN, nz), *vals = alloc<u32>(SH_ARENA_PLAN, nz);
      if (nz) be.for_each("shard_keys", nz, FShIota{keys, vals, c.rank});
      set_top(L_ZONE, keys, vals, nz);
    }
    {  // records: destination masks (a record can be needed on several shards), then the (destination, record) list
      u32 *mask = alloc<u32>(SH_ARENA_PLAN, A.n_records);
      be.fill32(mask, 0, (size_t)A.n_records + 1);
      if (A.n_values) be.for_each("shard_rec_mask", A.n_values, FShRecMask{S, W, val_dest, mask});
      mask_top(L_REC, mask, A.n_records);
    }
    plan_finish(meta, send_bytes);
  }
  // mask[row] = set of destinations (bits below G) -> top-level selection of level l: rows by (destination, row), a row once per
  // destination.  No sort: the tiles are in row order and the counts are laid out destination-major.
  void mask_top(int l, const u32 *mask, u32 n_rows) {
    const u32 T = (n_rows + SH_MASK_TILE - 1) / SH_MASK_TILE;
    u32 *counts = alloc<u32>(SH_ARENA_PLAN, (size_t)G * T + 1);
    be.fill32(counts + (size_t)G * T, 0, 1);
    if (T) be.for_each("shard_mask_count", T, FShMaskCount{mask, n_rows, G, T, counts});
    be.exclusive_scan(counts, G * T + 1);
    u32 nu = 0;
    be.download(&nu, counts + (size_t)G * T, 4);
    u32 *sel = alloc<u32>(SH_ARENA_PLAN, nu);
    if (T && nu) be.for_each("shard_mask_fill", T, FShMaskFill{mask, n_rows, G, T, counts, sel});
    active[l] = true;
    plan[l].multi = true;
    plan[l].sel = sel;
    plan[l].cap = nu;
    plan[l].m = m_dev(l);
    plan[l].row_off = row_off_dev(l);
    plan[l].slab_off = slab_off_dev(l);
    be.for_each("shard_bounds", G + 1, FShMaskBounds{counts, G, T, plan[l].row_off, plan[l].m});
  }

  // ---- pack the current plan into `send` (n_ranks blobs back to back, sizes as reported by the route call)
  void pack(u8 *send) {
    u64 blob_base[SH_MAX_RANKS + 1] = {0};
    u8 *bases[SH_MAX_RANKS] = {};
    for (u32 d = 0; d < G; d++) {
      u64 row[GAR_SHARD_META_WORDS] = {0};
      for (int l = 0; l < L_NLEVELS; l++) {
        row[l] = h_row_off[l][d + 1] - h_row_off[l][d];
        row[L_NLEVELS + l] = h_slab_off[l][d + 1] - h_slab_off[l][d];
      }
      blob_base[d + 1] = blob_base[d] + blob_bytes(row);
      bases[d] = send + blob_base[d];
    }
    pack_to(bases);
  }
  // The pack kernels with one destination address per rank: bases[d] = where this rank's blob for rank d starts: the send
  // buffer, or with peer memory mapped (gar_shard_pack_peers) this rank's own receive arena for its own blob and a local stage
  // for the others, which the engine then pushes to the other GPUs.
  // `level_done(l, end)` (optional) runs on the host after level l's kernels are queued; end[d] = bytes of destination d's blob
  // that are complete once those kernels have run — the engine uses it to start moving finished levels while later ones pack.
  template <class Done>
  void pack_to(u8 *const bases[SH_MAX_RANKS], Done level_done) {
    u64 lvl_off[SH_MAX_RANKS] = {0};
    u32 *any_long = alloc<u32>(SH_ARENA_PLAN, 1);
    be.fill32(any_long, 0, 1);
    for (int l = 0; l < L_NLEVELS; l++) {
      PackDst D{};
      for (u32 d = 0; d < G; d++) {
        u64 n = h_row_off[l][d + 1] - h_row_off[l][d], sb = h_slab_off[l][d + 1] - h_slab_off[l][d];
        D.base[d] = bases[d];
        D.lay[d] = level_layout(l, lvl_off[d], n, sb);
        lvl_off[d] = D.lay[d].end;
      }
      u32 m = h_row_off[l][G];
      if (!active[l] || !m) continue;
      be.for_each("shard_pack_rows", m, FShPackRows{src[l], SH_SCHEMA[l], plan[l], G, D, any_long});
      if (SH_SCHEMA[l].n_str && h_slab_off[l][G])
        be.for_each("shard_pack_long", SH_LONG_WORKERS, FShPackLong{src[l], SH_SCHEMA[l].n_str, plan[l], G, m, D, any_long});
      level_done(l, (const u64 *)lvl_off);
    }
    level_done((int)L_NLEVELS, (const u64 *)lvl_off);
  }
  void pack_to(u8 *const bases[SH_MAX_RANKS]) {
    pack_to(bases, [](int, const u64 *) {});
  }

  // ---- merge one level out of received blobs.  `from[s]` = (blob start, its meta row, level inside that blob).
  struct Seg {
    const u8 *blob;
    const u64 *meta;
    int lvl;
  };
  struct Merged {
    u32 n = 0;
    gar_str *str[SH_MAX_STR] = {};
    u8 *u8c[SH_MAX_U8] = {};
    u32 *u32c[SH_MAX_U32] = {};
    u32 *gid = nullptr;
    u32 *begin[SH_MAX_CHILD] = {};  // CSR begins (scanned), [n+1]
  };
  static LevelLayout layout_in_blob(const u64 *meta, int lvl) {
    u64 p = 0;
    LevelLayout L{};
    for (int l = 0; l <= lvl; l++) {
      L = level_layout(l, p, meta[l], meta[L_NLEVELS + l]);
      p = L.end;
    }
    return L;
  }
  // String bytes are NOT moved when `origin` is set: a merged string reference is the byte's distance from `origin`, one
  // address below every received blob, i.e. the receive buffers themselves serve as the slab of the merged tables (they must
  // stay untouched until the last diff of this exchange).  Copy mode (origin == nullptr; buffers further apart than a 40-bit
  // offset reaches, or GAR_SHARD_COPY_MERGE=1): the segments' bytes are appended to `slab`, *slab_used advances.
  Merged merge_level(int arena, int schema_lvl, const std::vector<Seg> &from, u8 *slab, u64 *slab_used, const u8 *origin = nullptr) {
    const LevelSchema &Sc = SH_SCHEMA[schema_lvl];
    Merged M;
    FShUnpackCols f{};
    f.nseg = (int)from.size();
    f.S = Sc;
    u32 n = 0;
    for (int s = 0; s < f.nseg; s++) {
      const Seg &g = from[s];
      f.seg[s].base = g.blob;
      f.seg[s].lay = layout_in_blob(g.meta, g.lvl);
      for (int c = 0; c < SH_MAX_CHILD; c++) f.has_cnt[s][c] = c < SH_SCHEMA[g.lvl].n_child;
      f.seg_row[s] = n;
      u64 sb = g.meta[L_NLEVELS + g.lvl];
      if (origin) {
        f.slab_base[s] = (u64)((g.blob + f.seg[s].lay.slab) - origin);
      } else {
        f.slab_base[s] = *slab_used;
        if (sb) be.copy_bytes(slab + *slab_used, g.blob + f.seg[s].lay.slab, sb);
        *slab_used += sb;
      }
      n += (u32)g.meta[g.lvl];
    }
    f.seg_row[f.nseg] = n;
    M.n = n;
    for (int c = 0; c < Sc.n_str; c++) f.D.str[c] = M.str[c] = alloc<gar_str>(arena, n);
    for (int c = 0; c < Sc.n_u8; c++) f.D.u8c[c] = M.u8c[c] = alloc<u8>(arena, n);
    for (int c = 0; c < Sc.n_u32; c++) f.D.u32c[c] = M.u32c[c] = alloc<u32>(arena, n);
    if (Sc.has_gid) f.D.gid = M.gid = alloc<u32>(arena, n);
    for (int c = 0; c < Sc.n_child; c++) {
      f.D.cnt[c] = M.begin[c] = alloc<u32>(arena, (size_t)n + 1);
      be.fill32(M.begin[c] + n, 0, 1);
    }
    if (n && f.nseg) be.for_each("shard_unpack_columns", n, f);
    for (int c = 0; c < Sc.n_child; c++) be.exclusive_scan(M.begin[c], n + 1);
    return M;
  }
  u64 slab_total(const std::vector<std::vector<Seg>> &groups) {
    u64 t = 0;
    for (auto &g : groups)
      for (auto &s : g) t += s.meta[L_NLEVELS + s.lvl];
    return t;
  }
  u64 recv_bytes(const u64 (*meta)[GAR_SHARD_META_WORDS]) {
    u64 t = 0;
    for (u32 s = 0; s < G; s++) t += blob_bytes(meta[s]);
    return t;
  }
  std::vector<Seg> segs(const u8 *recv, const u64 (*meta)[GAR_SHARD_META_WORDS], int lvl) {
    std::vector<Seg> v;
    u64 off = 0;
    for (u32 s = 0; s < G; s++) {
      v.push_back(Seg{recv + off, meta[s], lvl});
      off += blob_bytes(meta[s]);
    }
    return v;
  }

  // ---- after the round-1 exchange: build the directory tables (LBs, stubs, probes routed here)
  int unpack1(const u8 *recv, const u64 *meta_in) {
    recv1 = recv;
    for (u32 s = 0; s < G; s++)
      for (int w = 0; w < GAR_SHARD_META_WORDS; w++) meta1[s][w] = meta_in[(size_t)s * GAR_SHARD_META_WORDS + w];
    for (u32 s = 0; s < G; s++)
      if (meta1[s][SH_META_ZONE_FP] != zone_fp) {
        contract_error = "sharded mode: the zone table (zone_name, order, count) must be identical on every rank";
        return GAR_E_SHARD_CONTRACT;
      }
    be.shard_reset(SH_ARENA_DIR);
    auto lb = segs(recv, meta1, L_LB), st = segs(recv, meta1, L_STUB), stt = segs(recv, meta1, L_STUBTAG), pr = segs(recv, meta1, L_PROBE);
    u64 a_bytes = slab_total({lb, st, stt}), o_bytes = slab_total({pr});
    const u8 *origin = copy_merge ? nullptr : recv;
    u8 *aslab = nullptr, *oslab = nullptr;
    if (origin) {  // the received blobs are the slab (the caller keeps GAR_SLAB_PAD readable bytes behind them)
      aslab = oslab = (u8 *)origin;
      a_bytes = o_bytes = recv_bytes(meta1);
    } else {
      aslab = alloc<u8>(SH_ARENA_DIR, a_bytes + GAR_SLAB_PAD);
      oslab = alloc<u8>(SH_ARENA_DIR, o_bytes + GAR_SLAB_PAD);
      be.fill32((u32 *)(aslab + (a_bytes & ~(u64)3)), 0, GAR_SLAB_PAD / 4);
      be.fill32((u32 *)(oslab + (o_bytes & ~(u64)3)), 0, GAR_SLAB_PAD / 4);
    }
    u64 au = 0, ou = 0;
    Merged mlb = merge_level(SH_ARENA_DIR, L_LB, lb, aslab, &au, origin);
    Merged mst = merge_level(SH_ARENA_DIR, L_STUB, st, aslab, &au, origin);
    Merged mtt = merge_level(SH_ARENA_DIR, L_STUBTAG, stt, aslab, &au, origin);
    Merged mpr = merge_level(SH_ARENA_DIR, L_PROBE, pr, oslab, &ou, origin);
    Dt = DevTables{};
    Dt.cluster = S.cluster;
    Dt.cluster_len = S.cluster_len;
    gar_objects &O = Dt.o;
    O.n_objects = 0;
    u32 *zero3 = alloc<u32>(SH_ARENA_DIR, 4);
    be.fill32(zero3, 0, 4);
    O.obj_ann_begin = O.obj_lbi_begin = O.obj_port_begin = zero3;
    O.n_lbi = mpr.n;
    O.lbi_hostname = mpr.str[0];
    O.slab = oslab;
    O.slab_len = o_bytes;
    gar_actual &A = Dt.a;
    A.n_lbs = mlb.n;
    A.lb_region = mlb.str[0]; A.lb_name = mlb.str[1]; A.lb_dns = mlb.str[2]; A.lb_arn = mlb.str[3]; A.lb_state = mlb.u8c[0];
    A.n_accels = mst.n;
    A.acc_name = mst.str[0]; A.acc_dns = mst.str[1]; A.acc_enabled = mst.u8c[0];
    A.acc_tag_begin = mst.begin[0];
    u32 *nolis = alloc<u32>(SH_ARENA_DIR, (size_t)mst.n + 1);
    be.fill32(nolis, 0, (size_t)mst.n + 1);
    A.acc_lis_begin = nolis;
    A.n_tags = mtt.n;
    A.tag_key = mtt.str[0]; A.tag_val = mtt.str[1];
    A.lis_pr_begin = A.lis_eg_begin = A.eg_ep_begin = A.zone_rec_begin = A.rec_val_begin = zero3;
    A.slab = aslab;
    A.slab_len = a_bytes;
    dir_home = mpr.u32c[0];
    dir_lb_gid = mlb.gid;
    dir_stub_gid = mst.gid;
    return GAR_OK;
  }

  // ---- round 2: resolve the probes, route the answers to their homes
  void route2(u64 *meta, u64 *send_bytes) {
    delete dir_pipe;
    dir_pipe = new Pipeline<B>(be, Dt);
    dir_pipe->prepare_directory();
    const Work &W = dir_pipe->W;
    const gar_actual &A = Dt.a;
    plan_begin();
    LevelSrc x{};
    x.str[0] = A.lb_region; x.str[1] = A.lb_name; x.str[2] = A.lb_dns; x.str[3] = A.lb_arn; x.u8c[0] = A.lb_state; x.gid = dir_lb_gid;
    x.slab = A.slab; x.n = A.n_lbs; src[L_LB] = x;
    x = LevelSrc{}; x.str[0] = A.acc_name; x.str[1] = A.acc_dns; x.u8c[0] = A.acc_enabled; x.gid = dir_stub_gid; x.child_begin[0] = A.acc_tag_begin;
    x.slab = A.slab; x.n = A.n_accels; src[L_STUB] = x;
    x = LevelSrc{}; x.str[0] = A.tag_key; x.str[1] = A.tag_val; x.slab = A.slab; x.n = A.n_tags; src[L_STUBTAG] = x;
    u32 np = Dt.o.n_lbi;
    u32 *lb_mask = alloc<u32>(SH_ARENA_PLAN, A.n_lbs), *stub_mask = alloc<u32>(SH_ARENA_PLAN, A.n_accels);
    be.fill32(lb_mask, 0, (size_t)A.n_lbs + 1);
    be.fill32(stub_mask, 0, (size_t)A.n_accels + 1);
    if (np) be.for_each("shard_answer_probes", np, FShAnswer{Dt, W, dir_home, lb_mask, stub_mask});
    mask_top(L_LB, lb_mask, A.n_lbs);
    mask_top(L_STUB, stub_mask, A.n_accels);
    plan_finish(meta, send_bytes);
  }

  // ---- after the round-2 exchange: assemble the home sub-snapshot
  int unpack2(const u8 *recv2, const u64 *meta_in2) {
    u64 meta2[SH_MAX_RANKS][GAR_SHARD_META_WORDS];
    for (u32 s = 0; s < G; s++)
      for (int w = 0; w < GAR_SHARD_META_WORDS; w++) meta2[s][w] = meta_in2[(size_t)s * GAR_SHARD_META_WORDS + w];
    be.shard_reset(SH_ARENA_HOME);
    auto r1 = [&](int l) { return segs(recv1, meta1, l); };
    auto r2 = [&](int l) { return segs(recv2, meta2, l); };
    auto cat = [](std::vector<Seg> a, const std::vector<Seg> &b) {
      a.insert(a.end(), b.begin(), b.end());
      return a;
    };
    std::vector<Seg> s_obj = r1(L_OBJ), s_ann = r1(L_ANN), s_lbi = r1(L_LBI), s_port = r1(L_PORT);
    std::vector<Seg> s_acc = cat(r1(L_ACC), r2(L_STUB)), s_tag = cat(r1(L_TAG), r2(L_STUBTAG));
    std::vector<Seg> s_lis = r1(L_LIS), s_pr = r1(L_PR), s_eg = r1(L_EG), s_ep = r1(L_EP), s_rec = r1(L_REC), s_val = r1(L_VAL), s_zone = r1(L_ZONE);
    std::vector<Seg> s_lb = r2(L_LB);
    u64 o_bytes = slab_total({s_obj, s_ann, s_lbi, s_port});
    u64 a_bytes = slab_total({s_acc, s_tag, s_lis, s_pr, s_eg, s_ep, s_rec, s_val, s_zone, s_lb});
    // both receive buffers under one 40-bit string offset: no string byte moves
    const u8 *origin = recv1 < recv2 ? recv1 : recv2;
    const u8 *e1 = recv1 + recv_bytes(meta1), *e2 = recv2 + recv_bytes(meta2);
    const u64 span = (u64)((e1 > e2 ? e1 : e2) - origin);
    if (copy_merge || span + GAR_SLAB_PAD >= (1ull << 40)) origin = nullptr;
    u8 *oslab = nullptr, *aslab = nullptr;
    if (origin) {
      oslab = aslab = (u8 *)origin;
      o_bytes = a_bytes = span;
    } else {
      oslab = alloc<u8>(SH_ARENA_HOME, o_bytes + GAR_SLAB_PAD);
      aslab = alloc<u8>(SH_ARENA_HOME, a_bytes + GAR_SLAB_PAD);
      be.fill32((u32 *)(oslab + (o_bytes & ~(u64)3)), 0, GAR_SLAB_PAD / 4);
      be.fill32((u32 *)(aslab + (a_bytes & ~(u64)3)), 0, GAR_SLAB_PAD / 4);
    }
    u64 ou = 0, au = 0;
    const int AR = SH_ARENA_HOME;
    auto ml = [&](int lvl, const std::vector<Seg> &from, bool obj_side) { return merge_level(AR, lvl, from, obj_side ? oslab : aslab, obj_side ? &ou : &au, origin); };
    Merged obj = ml(L_OBJ, s_obj, true), ann = ml(L_ANN, s_ann, true);
    Merged lbi = ml(L_LBI, s_lbi, true), port = ml(L_PORT, s_port, true);
    u32 n_own = 0;
    for (u32 s = 0; s < G; s++) n_own += (u32)meta1[s][L_ACC];
    Merged acc = ml(L_ACC, s_acc, false), tag = ml(L_TAG, s_tag, false);
    Merged lis = ml(L_LIS, s_lis, false), pr = ml(L_PR, s_pr, false);
    Merged eg = ml(L_EG, s_eg, false), ep = ml(L_EP, s_ep, false);
    Merged rec = ml(L_REC, s_rec, false), val = ml(L_VAL, s_val, false);
    Merged zone = ml(L_ZONE, s_zone, false), lb = ml(L_LB, s_lb, false);

    H = DevTables{};
    H.cluster = S.cluster;
    H.cluster_len = S.cluster_len;
    gar_objects &O = H.o;
    O.n_objects = obj.n;
    O.obj_kind = obj.u8c[0]; O.obj_spec_type = obj.u8c[1]; O.obj_flags = obj.u8c[2];
    gar_str *ns = alloc<gar_str>(AR, obj.n), *nm = alloc<gar_str>(AR, obj.n);
    if (obj.n) be.for_each("shard_obj_ns_name", obj.n, FShObjNsName{obj.str[0], obj.u32c[0], ns, nm});
    O.obj_ns = ns; O.obj_name = nm; O.obj_ingress_class = obj.str[1];
    O.obj_ann_begin = obj.begin[0]; O.obj_lbi_begin = obj.begin[1]; O.obj_port_begin = obj.begin[2];
    O.n_ann = ann.n; O.ann_key = ann.str[0]; O.ann_val = ann.str[1];
    O.n_lbi = lbi.n; O.lbi_hostname = lbi.str[0];
    O.n_ports = port.n; O.port_number = (const i32 *)port.u32c[0]; O.port_proto = port.str[0];
    O.slab = oslab; O.slab_len = o_bytes;
    gar_actual &A = H.a;
    A.n_lbs = lb.n; A.lb_region = lb.str[0]; A.lb_name = lb.str[1]; A.lb_dns = lb.str[2]; A.lb_arn = lb.str[3]; A.lb_state = lb.u8c[0];
    A.n_accels = acc.n; A.acc_name = acc.str[0]; A.acc_dns = acc.str[1]; A.acc_enabled = acc.u8c[0];
    A.acc_tag_begin = acc.begin[0]; A.acc_lis_begin = acc.begin[1];
    A.n_tags = tag.n; A.tag_key = tag.str[0]; A.tag_val = tag.str[1];
    A.n_listeners = lis.n; A.lis_proto = lis.u8c[0]; A.lis_pr_begin = lis.begin[0]; A.lis_eg_begin = lis.begin[1];
    A.n_port_ranges = pr.n; A.pr_from = (const i32 *)pr.u32c[0];
    A.n_egs = eg.n; A.eg_ep_begin = eg.begin[0];
    A.n_endpoints = ep.n; A.ep_id = ep.str[0];
    A.n_zones = zone.n; A.zone_name = zone.str[0];
    u32 *zb = alloc<u32>(AR, (size_t)zone.n + 1);
    u32 *bad = alloc<u32>(AR, 2);
    be.fill32(bad, 0, 2);
    if (rec.n) be.for_each("shard_check_zone_order", rec.n, FShCheckZoneOrder{rec.u32c[0], zone.n, bad});
    u32 nbad = 0;
    be.download(&nbad, bad, 4);
    if (nbad) {
      contract_error = "sharded mode: a rank must hold the record sets of whole zones, zone ranges ascending with the rank";
      return GAR_E_SHARD_CONTRACT;
    }
    be.for_each("shard_zone_begin", zone.n + 1, FShZoneBegin{rec.u32c[0], rec.n, zb});
    A.zone_rec_begin = zb;
    A.n_records = rec.n; A.rec_name = rec.str[0]; A.rec_alias_dns = rec.str[1]; A.rec_type = rec.u8c[0]; A.rec_has_alias = rec.u8c[1];
    A.rec_val_begin = rec.begin[0];
    A.n_values = val.n; A.val_value = val.str[0];
    A.slab = aslab; A.slab_len = a_bytes;
    gids = ShGids{obj.gid, lb.gid, acc.gid, lis.gid, eg.gid, rec.gid, val.gid};
    guest_from = n_own;
    return GAR_OK;
  }
};
