// gar_pipeline.h — the diff as a sequence of data-parallel stages over a Backend.
//
// Backend = how a stage runs: the CUDA backend (gar_engine.cu) launches sm_100a kernels on a stream; the
// host-simulation backend (tests/hostsim) runs the same functors in loops so the CPU-only test tier can
// exercise the device logic.  Stages, functors and their order live here once.
//
// Backend interface:
//   template <class F> void for_each(const char *name, u32 n, const F &f);  // f(i) for i in [0, n)
//   template <class F> void for_each_warp(const char *name, u32 n, const F &f);  // f(i, i < n) for i in [0, roundup(n, 32)):
//                                                                                // full warps, f may use GAR_ANY votes
//   void exclusive_scan(u32 *data, u32 n);                                  // in place
//   void sort_pairs(u32 *keys, u32 *vals, u32 *keys_alt, u32 *vals_alt, u32 n, int bits);  // stable, result in keys/vals
//   void fill32(u32 *p, u32 value, size_t n);
//   void *ensure(int slot, size_t bytes);                                   // scratch buffer `slot`, at least `bytes`
//   void for_each_staged(const char *name, u32 n, const FTokenise &f);      // f(i) for i in [0, n); the CUDA backend stages
//                                                                           //   each block's hostnames in shared memory first
//   template <class... Fs> void for_each_multi(const char *name, std::initializer_list<u32> ns, const Fs &...fs);  // ONE launch: fs[k](i), i < ns[k]
//   template <class F> void for_each_dyn(const char *name, const u32 *n_dev, u32 cap, const F &f);       // f(i) for i < min(*n_dev, cap); the count
//   template <class F> void for_each_warp_dyn(const char *name, const u32 *n_dev, u32 cap, const F &f);  //   lives on the device: no read-back
//   void download(void *host_dst, const void *dev_src, size_t bytes);       // blocking
//   int graph_begin(u64 signature);  void graph_end();                      // launch-sequence caching (CUDA graphs): 0 = run the
//                                                                           // launches, 1 = run them while they are recorded, 2 = replayed
//   void download_start(int id, const void *dev_src, size_t bytes);         // id 0..1: small read-back in flight while later
//   void download_wait(int id, void *host_dst, size_t bytes);               //   stages are queued; wait blocks only if needed
#pragma once

#include <stdio.h>
#include <stdlib.h>

#include <initializer_list>

#include "gar_rows.h"

#if defined(__CUDA_ARCH__)
#define GAR_ATOMIC_ADD(p, v) atomicAdd((p), (v))
#else
#define GAR_ATOMIC_ADD(p, v) (*(p) += (v))
#endif

// ------------------------------------------------------------------ scratch slots

enum Slot {
  S_DERIVED, S_OFLAGS, S_OKEY_HASH, S_STAGE_GA, S_STAGE_R53, S_ANN_R53, S_ANN_NAME, S_ANN_TAGS, S_ANN_LISTEN, S_DPORT_BEGIN, S_DPORTS,
  S_TOK_CODE, S_TOK_NAME, S_TOK_REGION,
  S_ACC_FLAGS, S_ACC_OWNER_KEY, S_ACC_OWNER, S_ACC_THOST, S_ACC_MANAGED, S_ACC_OWNER_HASH, S_ACC_THOST_HASH, S_REC_NAME_HASH, S_VAL_KEY_HASH,
  S_REC_ZONE, S_VAL_REC, S_VAL_CLS, S_VAL_KEY, S_VAL_ORPHAN, S_VAL_LINK, S_ACC_DIGEST,
  S_R53_MODE, S_R53_ACC, S_R53_ACC_DNS, S_PAIR_BEGIN, S_PAIR_OBJ, S_PAIR_HN, S_PAIR_CODE, S_PAIR_ZONE, S_PAIR_REC,
  S_IX_LB, S_IX_OWNER = S_IX_LB + 3, S_IX_THOST = S_IX_OWNER + 3, S_IX_ZONE = S_IX_THOST + 3, S_IX_VAL = S_IX_ZONE + 3,
  S_IX_ALIAS = S_IX_VAL + 3, S_IX_OBJ = S_IX_ALIAS + 3, S_IX_OVN = S_IX_OBJ + 3,
  S_SORT_KEYS = S_IX_OVN + 3, S_SORT_VALS, S_SORT_KEYS_ALT, S_SORT_VALS_ALT, S_SORT_TAGS,
  S_COUNTS, S_STATUS_GA, S_STATUS_R53, S_OPS, S_ERRFLAG, S_IX_EG, S_IX_EG_ENT, S_IX_EG_PAD, S_ACC_CLAIMED,
  S_IXA_BEGIN, S_IXA_FILL, S_IXA_ENT, S_IXA_MULTI, S_OVN_FILL, S_OVN_MULTI, S_LB_HASH, S_REC_FLAGS,
  S_NSLOTS
};

// ------------------------------------------------------------------ functors (one per stage)

struct FClassify {
  DevTables T;
  Work W;
  u32 *derived_public;
  u8 *oflags;
  u32 *errflag;
  GAR_HD void operator()(u32 i) const {
    classify_object(T, W, i);
    u32 dv = W.derived[i];
    if (dv & OBJ_KEY_BAD) GAR_ATOMIC_ADD(errflag, 1u);
    derived_public[i] = dv & 0xFFu;
  }
};
// tokenise_hostnames is the one row pass whose strings are staged on chip (gar_engine.cu k_tokenise_staged): measured faster
// on the B200 than direct loads (DESIGN.md §5); staging measured slower for prepare_records.
struct FTokenise {
  DevTables T;
  Work W;
  GAR_HD void operator()(u32 i) const { tokenise_hostname(T, W, i); }
};
struct FDigestAccel {
  DevTables T;
  Work W;
  GAR_HD void operator()(u32 i) const { digest_accelerator(T, W, i); }
};
// child row -> parent row for a CSR (binary search on the begin array)
struct FExpand {
  const u32 *begin;
  u32 nparents;
  u32 *parent_of;
  GAR_HD void operator()(u32 c) const {
    u32 lo = 0, hi = nparents;  // last p with begin[p] <= c
    while (hi - lo > 1) {
      u32 mid = (lo + hi) >> 1;
      if (begin[mid] <= c) lo = mid;
      else hi = mid;
    }
    parent_of[c] = lo;
  }
};
// record row -> zone row, the hash of the record name (every (zone, name) key is derived from it), and its values: value ->
// record, owner-value classification.  One pass over the record table: a record's name and values are neighbours in the slab,
// so they share DRAM sectors.  A record set with MANY values (one hot TXT name claimed by thousands of owners) is not walked
// by its one thread: it goes on a list that FClassifyBigRecords works through with whole blocks.
constexpr u32 REC_INLINE_VALUES = 32;   // more values than this: a whole block works on the record
constexpr u32 REC_HUGE_VALUES = 4096;   // more than this: the whole grid does
struct FPrepareRecord {
  DevTables T;
  Work W;
  u32 *big, *huge;  // [0] = count, then record rows
  GAR_HD void operator()(u32 r) const {
    u32 lo = 0, hi = T.a.n_zones;
    while (hi - lo > 1) {
      u32 mid = (lo + hi) >> 1;
      if (T.a.zone_rec_begin[mid] <= r) lo = mid;
      else hi = mid;
    }
    W.rec_zone[r] = lo;
    const Str nm = mkstr(T.a.slab, T.a.rec_name[r]);
    const u64 nh = gar_hash(nm);
    W.rec_name_hash[r] = nh;
    W.rec_flags[r] = find_byte(nm, 0, '\\') < nm.n ? 1 : 0;
    if (T.a.rec_has_alias[r]) ix_count(W.hist[IX_ALIAS], key_hash_zoned_h(lo, nh));
    u32 v0 = T.a.rec_val_begin[r], v1 = T.a.rec_val_begin[r + 1];
    if (v1 - v0 > REC_INLINE_VALUES) {
      u32 *list = v1 - v0 > REC_HUGE_VALUES ? huge : big;
#if defined(__CUDA_ARCH__)
      list[1 + atomicAdd(list, 1u)] = r;
#else
      list[1 + list[0]++] = r;
#endif
      return;
    }
    for (u32 v = v0; v < v1; v++) {
      W.val_rec[v] = r;
      classify_value(T, W, v);
    }
  }
};
// fixed grid of BIG_BLOCKS x 256 threads: block b takes big records b, b + BIG_BLOCKS, ... and its threads stride over the
// values; the (few) huge records are strided over by the whole grid
constexpr u32 BIG_BLOCKS = 592;  // 4 x 148 SMs
struct FClassifyBigRecords {
  DevTables T;
  Work W;
  const u32 *big, *huge;
  GAR_HD void operator()(u32 i) const {
    const u32 blk = i >> 8, tid = i & 255u, nbig = big[0], nhuge = huge[0];
    for (u32 k = blk; k < nbig; k += BIG_BLOCKS) {
      u32 r = big[1 + k];
      for (u32 v = T.a.rec_val_begin[r] + tid; v < T.a.rec_val_begin[r + 1]; v += 256) {
        W.val_rec[v] = r;
        classify_value(T, W, v);
      }
    }
    for (u32 k = 0; k < nhuge; k++) {
      u32 r = huge[1 + k];
      for (u32 v = T.a.rec_val_begin[r] + i; v < T.a.rec_val_begin[r + 1]; v += BIG_BLOCKS * 256) {
        W.val_rec[v] = r;
        classify_value(T, W, v);
      }
    }
  }
};
struct FJsonCount {
  DevTables T;
  Work W;
  GAR_HD void operator()(u32 i) const {
    u32 n = 0;
    if (W.derived[i] & GAR_DV_PORTS_FROM_ANN) {
      u32 stk[GAR_JSON_STACK_WORDS];
      int c = json_listen_ports(mkstr(T.o.slab, W.ann_listen[i]), nullptr, stk);
      n = c < 0 ? 0u : (u32)c;
    }
    W.dport_begin[i] = n;
  }
};
struct FJsonWrite {
  DevTables T;
  Work W;
  GAR_HD void operator()(u32 i) const {
    if (!(W.derived[i] & GAR_DV_PORTS_FROM_ANN)) return;
    if (W.dport_begin[i + 1] == W.dport_begin[i] || W.dport_begin[i + 1] > W.dport_cap) return;
    u32 stk[GAR_JSON_STACK_WORDS];
    json_listen_ports(mkstr(T.o.slab, W.ann_listen[i]), W.dports + W.dport_begin[i], stk);
  }
};

// --- index rows: one functor per index says whether a row is indexed, its key hash and its entry payload
// (payload conventions: gar_rows.h "index probes").  The key pass streams the table once (coalesced) and leaves a
// complete 32-byte entry per row; the build then only moves entries.
// (region, name) hash of every load balancer: the only index key that is not produced by a row-local pass anyway
struct FLbHash {
  DevTables T;
  Work W;
  GAR_HD void operator()(u32 i) const {
    u64 h = key_hash_lb(mkstr(T.a.slab, T.a.lb_region[i]), mkstr(T.a.slab, T.a.lb_name[i]));
    W.lb_hash[i] = h;
    ix_count(W.hist[IX_LB], h);
  }
};
struct FRowLb {
  DevTables T;
  Work W;
  GAR_HD bool make(u32 i, u64 *h, IdxEntry *e) const {
    *h = W.lb_hash[i];
    e->a0 = T.a.lb_state[i];
    e->a1 = 0;
    e->s0 = T.a.lb_name[i];
    e->s1 = T.a.lb_region[i];
    return true;
  }
};
struct FRowOwner {
  DevTables T;
  Work W;
  GAR_HD bool make(u32 i, u64 *h, IdxEntry *e) const {
    u32 fl = W.acc_flags[i];
    *h = W.acc_owner_hash[i];
    e->a0 = fl;
    e->a1 = 0;
    e->s0 = W.acc_owner_key[i];
    e->s1 = 0;
    return (fl & ACC_MINE) && (fl & ACC_OWNER_KEYED) && i < W.acc_guest_from;
  }
};
struct FRowThost {
  DevTables T;
  Work W;
  GAR_HD bool make(u32 i, u64 *h, IdxEntry *e) const {
    *h = W.acc_thost_hash[i];
    e->a0 = e->a1 = 0;
    e->s0 = W.acc_thost[i];
    e->s1 = T.a.acc_dns[i];
    return (W.acc_flags[i] & ACC_MINE) != 0 && (!W.sharded || i >= W.acc_guest_from);
  }
};
struct FRowZone {
  DevTables T;
  GAR_HD bool make(u32 i, u64 *h, IdxEntry *e) const {
    Str zn = mkstr(T.a.slab, T.a.zone_name[i]);
    bool valid = zn.n >= 1 && zn.p[zn.n - 1] == '.';
    *h = valid ? key_hash_str(substr(zn, 0, zn.n - 1)) : 0;
    e->a0 = e->a1 = 0;
    e->s0 = T.a.zone_name[i];
    e->s1 = 0;
    return valid;
  }
};
struct FZoneLenMask {
  DevTables T;
  Work W;
  unsigned long long *mask;  // [4]
  GAR_HD void operator()(u32 z) const {
    Str zn = mkstr(T.a.slab, T.a.zone_name[z]);
    if (zn.n < 1 || zn.p[zn.n - 1] != '.') return;  // not indexed (FRowZone)
    ix_count(W.hist[IX_ZONE], key_hash_str(substr(zn, 0, zn.n - 1)));
    u32 b = zn.n - 1 < 255 ? zn.n - 1 : 255;
#if defined(__CUDA_ARCH__)
    atomicOr(&mask[b >> 6], 1ull << (b & 63));
#else
    mask[b >> 6] |= 1ull << (b & 63);
#endif
  }
};
struct FRowVal {
  DevTables T;
  Work W;
  GAR_HD bool make(u32 v, u64 *h, IdxEntry *e) const {
    u32 cls = W.val_cls[v];
    *h = W.val_key_hash[v];
    if (cls == VAL_NOT_OWNER) return false;
    u32 rec = W.val_rec[v];
    u32 kind = (cls & VAL_OWNER_INGRESS) ? 1u : 0u;
    u32 bs = (W.rec_flags[rec] & 1) ? VALNAME_HAS_BACKSLASH : 0u;
    e->a0 = rec;
    e->a1 = W.rec_zone[rec] | bs | (kind << 31);
    e->s0 = W.val_key[v];
    e->s1 = T.a.rec_name[rec];
    return true;
  }
};
struct FRowAlias {
  DevTables T;
  Work W;
  GAR_HD bool make(u32 r, u64 *h, IdxEntry *e) const {
    *h = key_hash_zoned_h(W.rec_zone[r], W.rec_name_hash[r]);
    e->a0 = W.rec_zone[r];
    e->a1 = T.a.rec_type[r];
    e->s0 = T.a.rec_name[r];
    e->s1 = T.a.rec_alias_dns[r];
    return T.a.rec_has_alias[r] != 0;
  }
};
struct FRowObj {
  DevTables T;
  Work W;
  GAR_HD bool make(u32 i, u64 *h, IdxEntry *e) const {
    gar_str ns = T.o.obj_ns[i];
    *h = W.okey_hash[i];
    e->a0 = T.o.obj_kind[i];
    e->a1 = 0;
    e->s0 = GAR_STR(GAR_STR_OFF(ns), GAR_STR_LEN(ns) + 1 + GAR_STR_LEN(T.o.obj_name[i]));
    e->s1 = 0;
    return !(W.derived[i] & OBJ_KEY_BAD);
  }
};
struct FRowOvn {
  DevTables T;
  Work W;
  GAR_HD bool make(u32 v, u64 *h, IdxEntry *e) const {
    u32 rec = W.val_rec[v];
    *h = key_hash_zoned_h(W.rec_zone[rec], W.rec_name_hash[rec]);
    e->a0 = rec;
    e->a1 = W.rec_zone[rec];
    e->s0 = T.a.rec_name[rec];
    e->s1 = T.a.val_value[v];
    return W.val_orphan[v] != 0;
  }
};

// Index build.  Fast path: (1) idx_rows: per row, entry + bucket key + bucket histogram; (2) scan; (3) idx_place: every
// indexed row drops its entry into its bucket with an atomic cursor (any order); (4) idx_order: buckets with >= 2
// entries are sorted by row id, which makes the result identical to a stable sort.  Buckets larger than
// IDX_SMALL_BUCKET (a hot key / adversarial input) raise `overflow`; the pipeline then rebuilds with the stable
// radix sort (idx_gather).
constexpr u32 IDX_SMALL_BUCKET = 48;
template <class RowF>
struct FIdxRows {
  RowF rowf;
  u32 *keys, *vals;
  IdxEntry *tmp;
  u32 *counts;
  u32 mask, nb;
  GAR_HD void operator()(u32 i) const {
    u64 h = 0;
    IdxEntry e;
    bool valid = rowf.make(i, &h, &e);
    u32 k = valid ? hash_bucket(h, mask) : nb;  // rows that are not indexed carry the sentinel key nb
    keys[i] = k;
    if (vals) vals[i] = i;  // only the radix rebuild sorts (key, row) pairs
    if (valid) {
      e.tag = hash_tag(h);
      e.row = i;
      tmp[i] = e;
      GAR_ATOMIC_ADD(&counts[k], 1u);
    }
  }
};
struct FIdxPlace {
  const u32 *keys;
  u32 *cursor;  // [nb] starts as a copy of begin[]
  const IdxEntry *tmp;
  IdxEntry *ent;
  u32 nb;
  GAR_HD void operator()(u32 i) const {
    u32 k = keys[i];
    if (k == nb) return;
#if defined(__CUDA_ARCH__)
    u32 pos = atomicAdd(&cursor[k], 1u);
#else
    u32 pos = cursor[k]++;
#endif
    ent[pos] = tmp[i];
  }
};
struct FIdxOrder {
  const u32 *begin;
  IdxEntry *ent;
  u32 *overflow;
  GAR_HD void operator()(u32 b) const {
    u32 lo = begin[b], m = begin[b + 1] - lo;
    if (m < 2) return;
    if (m > IDX_SMALL_BUCKET) {
      GAR_ATOMIC_ADD(overflow, 1u);
      return;
    }
    for (u32 k = 1; k < m; k++) {  // insertion sort of 32-byte entries by row id, in place
      IdxEntry x = ent[lo + k];
      u32 j = k;
      while (j > 0 && ent[lo + j - 1].row > x.row) {
        ent[lo + j] = ent[lo + j - 1];
        j--;
      }
      if (j != k) ent[lo + j] = x;
    }
  }
};
struct FIdxGather {  // radix fallback: position p of the stable sorted order holds row vals[p]
  const u32 *vals;
  const u32 *nvalid;
  const IdxEntry *tmp;
  IdxEntry *ent;
  GAR_HD void operator()(u32 p) const {
    if (p < *nvalid) ent[p] = tmp[vals[p]];
  }
};
// One-pass build (the default): the row-local passes have already counted every bucket (Work::hist); after ONE scan over the
// concatenated bucket arrays of all indexes this pass builds each row's entry from columns and hashes that already exist and
// drops it straight into its bucket — no temporary entry, no key array.  A bucket's second entry puts the bucket on the
// `multi` list: only those buckets are ordered afterwards (by row id == stable).
template <class RowF>
struct FIdxPlaceDirect {
  RowF rowf;
  u32 *cursor;    // this index's slice of the cursor array (a copy of the scanned bucket array): one atomic yields the position
  IdxEntry *ent;  // shared entry array of the group
  u32 mask;
  GAR_HD void operator()(u32 i) const {
    u64 h = 0;
    IdxEntry e;
    if (!rowf.make(i, &h, &e)) return;
    const u32 k = hash_bucket(h, mask);
#if defined(__CUDA_ARCH__)
    const u32 pos = atomicAdd(&cursor[k], 1u);
#else
    const u32 pos = cursor[k]++;
#endif
    e.tag = hash_tag(h);
    e.row = i;
    ent[pos] = e;
  }
};
// buckets with two or more entries, compacted into a list (one pass over the scanned bucket array; the appends are aggregated
// per warp, so the shared counter sees one atomic per warp, not one per bucket)
struct FIdxMultiList {
  const u32 *begin;
  u32 *multi;  // [0] = count, then bucket ids
  GAR_HD void operator()(u32 b) const {
    const bool m = begin[b + 1] - begin[b] >= 2;
#if defined(__CUDA_ARCH__)
    const unsigned active = __activemask();
    const unsigned votes = __ballot_sync(active, m);
    if (!m) return;
    const unsigned lane = threadIdx.x & 31u;
    const int leader = __ffs(votes) - 1;
    u32 base = 0;
    if ((int)lane == leader) base = atomicAdd(multi, (u32)__popc(votes));
    base = __shfl_sync(votes, base, leader);
    multi[1 + base + __popc(votes & ((1u << lane) - 1u))] = b;
#else
    if (m) multi[1 + multi[0]++] = b;
#endif
  }
};
struct FIdxOrderMulti {
  const u32 *begin;  // the group's whole bucket array
  IdxEntry *ent;
  const u32 *multi;
  u32 *overflow;
  GAR_HD void operator()(u32 t) const {
    const u32 b = multi[1 + t];
    const u32 lo = begin[b], m = begin[b + 1] - lo;
    if (m > IDX_SMALL_BUCKET) {
      GAR_ATOMIC_ADD(overflow, 1u);
      return;
    }
    for (u32 k = 1; k < m; k++) {  // insertion sort of 32-byte entries by row id, in place
      IdxEntry x = ent[lo + k];
      u32 j = k;
      while (j > 0 && ent[lo + j - 1].row > x.row) {
        ent[lo + j] = ent[lo + j - 1];
        j--;
      }
      if (j != k) ent[lo + j] = x;
    }
  }
};
// everything the host reads back at the END of a diff, gathered into one small block (no read-back in the middle)
enum FlagWord { FW_BAD_KEYS = 0, FW_IDX_OVERFLOW = 1, FW_NDPORTS = 2, FW_NPAIRS = 3, FW_SEC0 = 4 /* 5 section words */, FW_WORDS = 16 };
struct FGatherFinal {
  const u32 *src;
  u32 idx[5];
  const u32 *npairs;  // nullable
  u32 *flags;
  GAR_HD void operator()(u32 k) const {
    if (k < 5) flags[FW_SEC0 + k] = src[idx[k]];
    else if (npairs) flags[FW_NPAIRS] = *npairs;
  }
};
struct FGather5 {
  const u32 *src;
  u32 idx[5];
  const u32 *extra;
  u32 *dst;
  GAR_HD void operator()(u32 k) const { dst[k] = k < 5 ? src[idx[k]] : *extra; }
};
#define GAR_RETRY_WITH_RADIX 1000  // Pipeline::run: rebuild with force_radix (not an error)
#define GAR_REFUSE_EMPTY_CACHE 1001  // orphan deletes against an empty object table (garecon.h "Orphan sweep precondition")
struct FGatherHeader {
  const u32 *ndports;
  u32 *flags;
  GAR_HD void operator()(u32) const { flags[FW_NDPORTS] = *ndports; }
};
// the two per-value joins in one pass (independent probe chains overlap): first alias record under the value's (zone, name),
// and whether the owner the value names is still in the object cache
struct FValueJoins {
  DevTables T;
  Work W;
  GAR_HD void operator()(u32 v) const {
    link_value_alias(T, W, v);
    mark_orphan_value(T, W, v);
  }
};

// --- count / emit.  counts layout: [GA obj: n][GA orphan: nacc][R53 obj: n][orphan alias: nrec][orphan value: nval][total]
struct CountLayout {
  u32 n, nacc, nrec, nval;
  GAR_HD u32 ga_obj(u32 i) const { return i; }
  GAR_HD u32 ga_orph(u32 a) const { return n + a; }
  GAR_HD u32 r53_obj(u32 i) const { return n + nacc + i; }
  GAR_HD u32 base0() const { return 2 * n + nacc; }
  GAR_HD u32 base1() const { return 2 * n + nacc + nrec; }
  GAR_HD u32 total() const { return 2 * n + nacc + nrec + nval; }
};
// Object sections: every object is evaluated ONCE.  The evaluation writes the status word, the op count and
// up to OPS_STAGE_CAP ops into the object's staging slot; after the scan FCompactOps moves staged ops to their
// final position (objects with more ops than the slot holds are re-evaluated straight into the output).
constexpr u32 OPS_STAGE_CAP = 4;
// `rows` (nullable) selects a subset of object rows (incremental mode): slot t evaluates object rows[t]; status, counts
// and staging are indexed by the slot, everything about the object by its row.
struct FGaObj {
  DevTables T;
  Work W;
  u32 *counts;    // [slots] this section's counts
  gar_op *stage;  // [slots * OPS_STAGE_CAP]
  u32 *status;
  const u32 *rows;
  GAR_HD void operator()(u32 t, bool valid) const {
    u32 i = (rows && valid) ? rows[t] : t;
    OpSink s{stage + (size_t)t * OPS_STAGE_CAP, 0, OPS_STAGE_CAP};
    u32 st = ga_reconcile(T, W, i, valid, s);
    if (valid) {
      status[t] = st;
      counts[t] = s.n;
    }
  }
};
struct FR53Obj {
  DevTables T;
  Work W;
  u32 *counts;
  gar_op *stage;
  u32 *status;
  const u32 *rows;
  GAR_HD void operator()(u32 t, bool valid) const {
    u32 i = (rows && valid) ? rows[t] : t;
    OpSink s{stage + (size_t)t * OPS_STAGE_CAP, 0, OPS_STAGE_CAP};
    // objects finished by r53_prepare keep the status it wrote; every other status is produced here
    u32 prev = (valid && W.r53_mode[i] == R53_MODE_DONE) ? status[t] : 0;
    u32 st = r53_combine(T, W, i, t, valid, prev, s);
    if (valid) {
      status[t] = st;
      counts[t] = s.n;
    }
  }
};
struct FR53Prepare {
  DevTables T;
  Work W;
  u32 *status;
  const u32 *rows;
  GAR_HD void operator()(u32 t, bool valid) const { r53_prepare(T, W, (rows && valid) ? rows[t] : t, t, valid, status); }
};
struct FR53FillPairs {
  DevTables T;
  Work W;
  const u32 *rows;
  GAR_HD void operator()(u32 t) const { r53_fill_pairs(T, W, rows ? rows[t] : t, t); }
};
struct FR53Pair {
  DevTables T;
  Work W;
  GAR_HD void operator()(u32 p, bool valid) const { r53_pair(T, W, p, valid); }
};
// incremental mode: processDelete of one work-queue key that left the cache (globalaccelerator/service.go:28-52,
// route53/service.go:29-46): cleanup of everything the key owns, in the reference's order
struct DelKeys {
  const u8 *kind;
  const gar_str *key;  // refs into `slab`
  const u8 *slab;
};
struct FDelKeyGa {
  DevTables T;
  Work W;
  DelKeys D;
  u32 *counts;   // count pass: written; emit pass: scanned
  gar_op *ops;   // nullptr in the count pass
  u32 cap;
  GAR_HD void operator()(u32 k) const {
    u32 kind = D.kind[k];
    Str key = mkstr(D.slab, D.key[k]);
    if (ops && counts[k + 1] > cap) return;  // beyond the buffer: dropped, the diff is re-run
    OpSink s{ops ? ops + counts[k] : nullptr, 0, 0xFFFFFFFFu};
    OwnerIter it = owner_open(W, key_hash_kinded(kind, key), key);
    for (u32 acc; (acc = owner_next(T, W, kind, it)) != GAR_NONE;) put_delete_chain(T, s, GAR_NONE, 0, acc);
    if (!ops) counts[k] = s.n;
  }
};
struct FDelKeyR53 {
  DevTables T;
  Work W;
  DelKeys D;
  u32 *counts;
  gar_op *ops;
  u32 cap;
  GAR_HD void operator()(u32 k) const {
    u32 kind = D.kind[k];
    Str key = mkstr(D.slab, D.key[k]);
    if (ops && counts[k + 1] > cap) return;
    OpSink s{ops ? ops + counts[k] : nullptr, 0, 0xFFFFFFFFu};
    Owned ow;
    owned_collect(T, W, key_hash_kinded(kind, key), kind, key, ow);
    r53_cleanup(T, W, GAR_NONE, 0, ow, s);
    if (!ops) counts[k] = s.n;
  }
};
struct FRowKnownEg {
  gar_bindings b;
  GAR_HD bool make(u32 i, u64 *h, IdxEntry *e) const {
    *h = gar_hash(mkstr(b.slab, b.known_eg_arn[i]));
    e->a0 = e->a1 = 0;
    e->s0 = b.known_eg_arn[i];
    e->s1 = 0;
    return true;
  }
};
struct FEgb {
  DevTables T;
  Work W;
  DevBindings B;
  u32 *counts;   // count pass: written; emit pass: scanned
  gar_op *ops;
  u32 *status;
  u32 cap;
  GAR_HD void operator()(u32 k) const {
    if (ops && counts[k + 1] > cap) return;
    OpSink s{ops ? ops + counts[k] : nullptr, 0, 0xFFFFFFFFu};
    u32 st = egb_reconcile(T, W, B, k, s);
    if (ops) status[k] = st;
    else counts[k] = s.n;
  }
};
struct FGatherDerived {
  const u32 *derived, *rows;
  u32 *out;
  GAR_HD void operator()(u32 t) const { out[t] = derived[rows[t]] & 0xFFu; }
};
struct FCompactOps {
  DevTables T;
  Work W;
  const u32 *scanned;  // exclusive-scanned counts of this section (entry t+1 exists: the layout is contiguous)
  const gar_op *stage;
  gar_op *ops;
  u32 ctrl;
  const u32 *rows;
  u32 cap;  // capacity of `ops`: nothing is written at or beyond it
  GAR_HD void operator()(u32 t, bool valid) const {
    u32 i = (rows && valid) ? rows[t] : t;
    u32 off = 0, c = 0;
    if (valid) {
      off = scanned[t];
      c = scanned[t + 1] - off;
      if (off > cap || c > cap - off) c = 0;  // does not fit: dropped (the total in the flag block tells the host)
      if (c <= OPS_STAGE_CAP)
        for (u32 k = 0; k < c; k++) ops[off + k] = stage[(size_t)t * OPS_STAGE_CAP + k];
    }
    // objects with more ops than a staging slot holds are re-evaluated straight into the output (warp-uniform:
    // the decide functions vote, so the whole warp enters when any lane needs it)
    bool redo = valid && c > OPS_STAGE_CAP;
    if (GAR_ANY(redo)) {
      OpSink s{ops + off, 0, redo ? c : 0u};
      if (ctrl == GAR_CTRL_GA) ga_reconcile(T, W, i, redo, s);
      else r53_reconcile(T, W, i, redo, s);  // the per-object routine: same decisions as prepare/pairs/combine
    }
  }
};
struct FGaOrphan {
  DevTables T;
  Work W;
  CountLayout L;
  u32 *counts;
  gar_op *ops;
  u32 cap;
  GAR_HD void operator()(u32 a) const {
    if (ops && counts[L.ga_orph(a) + 1] == counts[L.ga_orph(a)]) return;  // emit pass: nothing to write
    if (ops && counts[L.ga_orph(a) + 1] > cap) return;                    // beyond the buffer: dropped, the diff is re-run
    OpSink s{ops ? ops + counts[L.ga_orph(a)] : nullptr, 0, 0xFFFFFFFFu};
    ga_orphan(T, W, a, s);
    if (!ops) counts[L.ga_orph(a)] = s.n;
  }
};
// orphan section order: per zone, alias phase (by record row) then metadata phase (by value row)
struct FR53OrphanAlias {
  DevTables T;
  Work W;
  CountLayout L;
  u32 *counts;
  gar_op *ops;
  u32 cap;
  GAR_HD void operator()(u32 r) const {
    if (!ops) {
      OpSink s{nullptr, 0, 0};
      r53_orphan_alias(T, W, r, s);
      counts[L.base0() + r] = s.n;
      return;
    }
    if (counts[L.base0() + r + 1] == counts[L.base0() + r]) return;
    if (counts[L.total()] > cap) return;  // the R53 orphan section interleaves two count ranges: all or nothing
    u32 z = W.rec_zone[r];
    u32 zv = T.a.rec_val_begin[T.a.zone_rec_begin[z]];  // first value row of the zone
    u32 off = counts[L.base0()] + (counts[L.base1() + zv] - counts[L.base1()]) + (counts[L.base0() + r] - counts[L.base0()]);
    OpSink s{ops + off, 0, 0xFFFFFFFFu};
    r53_orphan_alias(T, W, r, s);
  }
};
struct FR53OrphanValue {
  DevTables T;
  Work W;
  CountLayout L;
  u32 *counts;
  gar_op *ops;
  u32 cap;
  GAR_HD void operator()(u32 v) const {
    if (!ops) {
      counts[L.base1() + v] = W.val_orphan[v];
      return;
    }
    if (!W.val_orphan[v] || counts[L.total()] > cap) return;
    u32 r = W.val_rec[v];
    u32 z = W.rec_zone[r];
    u32 rend = T.a.zone_rec_begin[z + 1];  // alias-phase ops of zones 0..z precede
    u32 off = counts[L.base0()] + (counts[L.base0() + rend] - counts[L.base0()]) + (counts[L.base1() + v] - counts[L.base1()]);
    gar_op o;
    o.head = GAR_OP_HEAD(GAR_OP_R53_DELETE_RECORD, GAR_CTRL_R53, 0);
    o.obj = GAR_NONE;
    o.sub = 1;
    o.a0 = z;
    o.a1 = r;
    o.a2 = v;
    ops[off] = o;
  }
};

// ------------------------------------------------------------------ the pipeline

struct DiffCounts {
  u64 n_ops;
  u64 section_begin[GAR_N_SECTIONS + 1];
  u64 n_dports;
  u32 bad_keys;
};

GAR_HD u32 next_pow2(u32 x) {
  u32 p = 1;
  while (p < x) p <<= 1;
  return p;
}
inline int ilog2(u32 p) {
  int b = 0;
  while ((1u << b) < p) b++;
  return b;
}

template <class B>
struct Pipeline {
  B &be;
  DevTables T;
  Work W{};
  bool force_radix = false;  // set when a bucket exceeded IDX_SMALL_BUCKET in the previous attempt
  explicit Pipeline(B &b, const DevTables &t) : be(b), T(t) {}

  // nb: buckets (power of two).  load: target rows per bucket used to size nb from the row count.
  template <class RowF>
  HashIdx build_index(int slot, u32 nrows, u32 load, RowF rowf, u32 *overflow, bool force_radix) {
    u32 nb = next_pow2(nrows / load < 16 ? 16 : nrows / load);
    u32 *keys = (u32 *)be.ensure(S_SORT_KEYS, sizeof(u32) * (size_t)(nrows + 1));
    u32 *vals = (u32 *)be.ensure(S_SORT_VALS, sizeof(u32) * (size_t)(nrows + 1));
    IdxEntry *tmp = (IdxEntry *)be.ensure(S_SORT_TAGS, sizeof(IdxEntry) * (size_t)(nrows + 1));
    u32 *begin = (u32 *)be.ensure(slot + 0, sizeof(u32) * (size_t)(nb + 2));
    IdxEntry *ent = (IdxEntry *)be.ensure(slot + 1, sizeof(IdxEntry) * (size_t)(nrows + 1));
    be.fill32(begin, 0, nb + 2);
    if (nrows) be.for_each("idx_rows", nrows, FIdxRows<RowF>{rowf, keys, force_radix ? vals : nullptr, tmp, begin, nb - 1, nb});
    be.exclusive_scan(begin, nb + 2);  // begin[b] = #rows with key < b; begin[nb] = #indexed rows
    if (nrows && !force_radix) {
      u32 *cursor = (u32 *)be.ensure(S_SORT_KEYS_ALT, sizeof(u32) * (size_t)(nb + 1));
      be.copy32(cursor, begin, nb);
      be.for_each("idx_place", nrows, FIdxPlace{keys, cursor, tmp, ent, nb});
      be.for_each("idx_order", nb, FIdxOrder{begin, ent, overflow});
    } else if (nrows) {
      u32 *keys2 = (u32 *)be.ensure(S_SORT_KEYS_ALT, sizeof(u32) * (size_t)(nrows + 1));
      u32 *vals2 = (u32 *)be.ensure(S_SORT_VALS_ALT, sizeof(u32) * (size_t)(nrows + 1));
      be.sort_pairs(keys, vals, keys2, vals2, nrows, ilog2(nb) + 1);
      be.for_each("idx_gather", nrows, FIdxGather{vals, begin + nb, tmp, ent});
    }
    return HashIdx{begin, ent, nb - 1};
  }

  // ---- prepare: everything that depends on the snapshot only (stages 1-3).  Runs once per loaded snapshot; the
  // digests and indexes stay resident for every later diff (full or incremental).
  bool prepared = false;
  u64 n_dports = 0;  // from the final read-back of the last diff
  u32 *errflag = nullptr;

  u32 acc_guest_from = 0xFFFFFFFFu;  // sharded mode: set before prepare()
  u32 sharded = 0;
  bool orphan_sweep = true;        // GAR_FLAG_NO_ORPHANS clears it
  bool allow_empty_cache = false;  // GAR_FLAG_ALLOW_EMPTY_CACHE

  void alloc_work() {
    const u32 n = T.o.n_objects, nlbi = T.o.n_lbi, nacc = T.a.n_accels, nrec = T.a.n_records, nval = T.a.n_values;
    W.derived = (u32 *)be.ensure(S_DERIVED, 4 * (size_t)(n + 1));
    W.okey_hash = (u64 *)be.ensure(S_OKEY_HASH, 8 * (size_t)(n + 1));
    W.ann_r53 = (gar_str *)be.ensure(S_ANN_R53, 8 * (size_t)(n + 1));
    W.ann_name = (gar_str *)be.ensure(S_ANN_NAME, 8 * (size_t)(n + 1));
    W.ann_tags = (gar_str *)be.ensure(S_ANN_TAGS, 8 * (size_t)(n + 1));
    W.ann_listen = (gar_str *)be.ensure(S_ANN_LISTEN, 8 * (size_t)(n + 1));
    W.dport_begin = (u32 *)be.out_dport_begin(n);
    W.tok_code = (u8 *)be.out_tok_code(nlbi);
    W.tok_name = (gar_str *)be.out_tok_name(nlbi);
    W.tok_region = (gar_str *)be.out_tok_region(nlbi);
    W.acc_flags = (u32 *)be.ensure(S_ACC_FLAGS, 4 * (size_t)(nacc + 1));
    W.acc_owner_key = (gar_str *)be.ensure(S_ACC_OWNER_KEY, 8 * (size_t)(nacc + 1));
    W.acc_owner = (gar_str *)be.ensure(S_ACC_OWNER, 8 * (size_t)(nacc + 1));
    W.acc_thost = (gar_str *)be.ensure(S_ACC_THOST, 8 * (size_t)(nacc + 1));
    W.acc_managed = (gar_str *)be.ensure(S_ACC_MANAGED, 8 * (size_t)(nacc + 1));
    W.acc_owner_hash = (u64 *)be.ensure(S_ACC_OWNER_HASH, 8 * (size_t)(nacc + 1));
    W.acc_thost_hash = (u64 *)be.ensure(S_ACC_THOST_HASH, 8 * (size_t)(nacc + 1));
    W.rec_name_hash = (u64 *)be.ensure(S_REC_NAME_HASH, 8 * (size_t)(nrec + 1));
    W.val_key_hash = (u64 *)be.ensure(S_VAL_KEY_HASH, 8 * (size_t)(nval + 1));
    W.rec_zone = (u32 *)be.ensure(S_REC_ZONE, 4 * (size_t)(nrec + 1));
    W.val_rec = (u32 *)be.ensure(S_VAL_REC, 4 * (size_t)(nval + 1));
    W.val_cls = (u8 *)be.ensure(S_VAL_CLS, nval + 1);
    W.val_key = (gar_str *)be.ensure(S_VAL_KEY, 8 * (size_t)(nval + 1));
    W.val_orphan = (u8 *)be.ensure(S_VAL_ORPHAN, nval + 1);
    W.val_link = (ValLink *)be.ensure(S_VAL_LINK, sizeof(ValLink) * (size_t)(nval + 1));
    W.acc_digest = (AccDigest *)be.ensure(S_ACC_DIGEST, sizeof(AccDigest) * (size_t)(nacc + 1));
    W.r53_mode = (u8 *)be.ensure(S_R53_MODE, (size_t)n + 1);
    W.r53_acc = (u32 *)be.ensure(S_R53_ACC, 4 * (size_t)(n + 1));
    W.r53_acc_dns = (gar_str *)be.ensure(S_R53_ACC_DNS, 8 * (size_t)(n + 1));
    W.lb_hash = (u64 *)be.ensure(S_LB_HASH, 8 * (size_t)(T.a.n_lbs + 1));
    W.rec_flags = (u8 *)be.ensure(S_REC_FLAGS, (size_t)nrec + 1);
    for (int k = 0; k < IX_N; k++) W.hist[k] = IxHist{nullptr, 0};
    W.pair_cap = 0;
    W.dport_cap = 0;
    errflag = (u32 *)be.ensure(S_ERRFLAG, 256);
    be.fill32(errflag, 0, FW_WORDS);
    W.acc_guest_from = acc_guest_from;
    W.sharded = sharded;
    W.acc_claimed = nullptr;
  }
  void stage1() {
    const u32 n = T.o.n_objects, nlbi = T.o.n_lbi, nacc = T.a.n_accels, nrec = T.a.n_records, nval = T.a.n_values;
    u32 *derived_public = (u32 *)be.out_derived(n);
    // stage 1: row-local preprocessing
    if (n) be.for_each("classify_objects", n, FClassify{T, W, derived_public, nullptr, errflag});
    if (nlbi) be.for_each_staged("tokenise_hostnames", nlbi, FTokenise{T, W});
    if (nacc) be.for_each("digest_accelerators", nacc, FDigestAccel{T, W});
    if (T.a.n_lbs) be.for_each("hash_load_balancers", T.a.n_lbs, FLbHash{T, W});
    {
      unsigned long long *zm = (unsigned long long *)(errflag + 16 + 8);  // 32 bytes inside the 256-byte flag block, 8-byte aligned
      be.fill32((u32 *)zm, 0, 8);
      if (T.a.n_zones) be.for_each("zone_len_mask", T.a.n_zones, FZoneLenMask{T, W, zm});
      W.zone_len_mask = (const u64 *)zm;
    }
    if (nrec) {  // includes the records' values
      u32 *big = (u32 *)be.ensure(S_SORT_KEYS, 4 * (size_t)(nval / REC_INLINE_VALUES + 2));
      u32 *huge = (u32 *)be.ensure(S_SORT_VALS, 4 * (size_t)(nval / REC_HUGE_VALUES + 2));
      be.fill32(big, 0, 1);
      be.fill32(huge, 0, 1);
      be.for_each("prepare_records", nrec, FPrepareRecord{T, W, big, huge});
      if (nval > REC_INLINE_VALUES) be.for_each("prepare_records", BIG_BLOCKS * 256, FClassifyBigRecords{T, W, big, huge});
    }
  }
  // ---- one-pass index build (the default).  plan: which indexes, their bucket counts and where each one's slice of the
  // shared bucket / entry arrays starts.  The histogram hooks (Work::hist) must be armed BEFORE the row-local passes run.
  struct IxPlan {
    u32 off[IX_N] = {}, nb[IX_N] = {}, rows[IX_N] = {};
    bool want[IX_N] = {};
    u32 total_nb = 0;
    u64 total_rows = 0;
  };
  IxPlan planA;
  u32 *ixa_begin = nullptr, *ixa_fill = nullptr, *ixa_multi = nullptr;
  IdxEntry *ixa_ent = nullptr;
  u32 ovn_nb = 0;
  void arm_group_a(u32 want_mask) {
    const u32 rows[IX_N] = {T.a.n_lbs, T.a.n_accels, T.a.n_accels, T.a.n_zones, T.a.n_values, T.a.n_records, T.o.n_objects, 0};
    const u32 load[IX_N] = {1, 1, 1, 1, 1, 2, 1, 8};
    planA = IxPlan{};
    for (int k = 0; k < IX_OVN; k++) {
      planA.want[k] = (want_mask >> k) & 1u;
      if (!planA.want[k]) continue;
      planA.rows[k] = rows[k];
      planA.nb[k] = next_pow2(rows[k] / load[k] < 16 ? 16 : rows[k] / load[k]);
      planA.off[k] = planA.total_nb;
      planA.total_nb += planA.nb[k];
      planA.total_rows += rows[k];
    }
    ixa_begin = (u32 *)be.ensure(S_IXA_BEGIN, 4 * (size_t)(planA.total_nb + 2));
    be.fill32(ixa_begin, 0, (size_t)planA.total_nb + 2);
    for (int k = 0; k < IX_OVN; k++)
      if (planA.want[k]) W.hist[k] = IxHist{ixa_begin + planA.off[k], planA.nb[k] - 1};
  }
  HashIdx group_a_index(int k) const { return HashIdx{ixa_begin + planA.off[k], ixa_ent, planA.nb[k] - 1}; }
  template <class RowF>
  FIdxPlaceDirect<RowF> placer(int k, RowF rowf) const {
    return FIdxPlaceDirect<RowF>{rowf, ixa_fill + planA.off[k], ixa_ent, planA.nb[k] - 1};
  }
  // scan + place + order of group A (after every armed row pass has run)
  void finish_group_a() {
    u32 *overflow = errflag + FW_IDX_OVERFLOW;
    be.exclusive_scan(ixa_begin, planA.total_nb + 1);  // positions in the shared entry array; [total_nb] = number of entries
    ixa_fill = (u32 *)be.ensure(S_IXA_FILL, 4 * (size_t)(planA.total_nb + 1));  // the placement cursors
    ixa_ent = (IdxEntry *)be.ensure(S_IXA_ENT, sizeof(IdxEntry) * (size_t)(planA.total_rows + 1));
    const u32 multi_cap = (u32)(planA.total_rows / 2 + 1);
    ixa_multi = (u32 *)be.ensure(S_IXA_MULTI, 4 * (size_t)(multi_cap + 2));
    be.copy32(ixa_fill, ixa_begin, (size_t)planA.total_nb + 1);
    be.fill32(ixa_multi, 0, 1);
    const IxPlan &P = planA;
    auto n = [&](int k) { return P.want[k] ? P.rows[k] : 0u; };
    be.for_each_multi("idx_place", {n(IX_LB), n(IX_OWNER), n(IX_THOST), n(IX_ZONE), n(IX_VAL), n(IX_ALIAS), n(IX_OBJ), P.total_nb},
                      placer(IX_LB, FRowLb{T, W}), placer(IX_OWNER, FRowOwner{T, W}), placer(IX_THOST, FRowThost{T, W}), placer(IX_ZONE, FRowZone{T}),
                      placer(IX_VAL, FRowVal{T, W}), placer(IX_ALIAS, FRowAlias{T, W}), placer(IX_OBJ, FRowObj{T, W}), FIdxMultiList{ixa_begin, ixa_multi});
    be.for_each_dyn("idx_order", ixa_multi, multi_cap, FIdxOrderMulti{ixa_begin, ixa_ent, ixa_multi, overflow});
    if (P.want[IX_LB]) W.ix_lb = group_a_index(IX_LB);
    if (P.want[IX_OWNER]) W.ix_owner = group_a_index(IX_OWNER);
    if (P.want[IX_THOST]) W.ix_thost = group_a_index(IX_THOST);
    if (P.want[IX_ZONE]) W.ix_zone = group_a_index(IX_ZONE);
    if (P.want[IX_VAL]) W.ix_val = group_a_index(IX_VAL);
    if (P.want[IX_ALIAS]) W.ix_alias = group_a_index(IX_ALIAS);
    if (P.want[IX_OBJ]) W.ix_obj = group_a_index(IX_OBJ);
  }
  // the orphan-value index: its keys exist only after the per-value joins (which count its buckets: mark_orphan_value)
  void arm_ovn() {
    ovn_nb = next_pow2(T.a.n_values / 8 < 16 ? 16 : T.a.n_values / 8);
    u32 *cnt = (u32 *)be.ensure(S_IX_OVN + 0, 4 * (size_t)(ovn_nb + 2));
    be.fill32(cnt, 0, (size_t)ovn_nb + 2);
    W.hist[IX_OVN] = IxHist{cnt, ovn_nb - 1};
  }
  void finish_ovn() {
    const u32 nval = T.a.n_values;
    u32 *begin = W.hist[IX_OVN].cnt;
    be.exclusive_scan(begin, ovn_nb + 1);
    u32 *cursor = (u32 *)be.ensure(S_OVN_FILL, 4 * (size_t)(ovn_nb + 1));
    IdxEntry *ent = (IdxEntry *)be.ensure(S_IX_OVN + 1, sizeof(IdxEntry) * (size_t)(nval + 1));
    u32 *multi = (u32 *)be.ensure(S_OVN_MULTI, 4 * (size_t)(nval / 2 + 3));
    be.copy32(cursor, begin, (size_t)ovn_nb + 1);
    be.fill32(multi, 0, 1);
    be.for_each_multi("idx_place", {nval, ovn_nb}, FIdxPlaceDirect<FRowOvn>{FRowOvn{T, W}, cursor, ent, ovn_nb - 1}, FIdxMultiList{begin, multi});
    be.for_each_dyn("idx_order", multi, nval / 2 + 1, FIdxOrderMulti{begin, ent, multi, errflag + FW_IDX_OVERFLOW});
    W.ix_ovn = HashIdx{begin, ent, ovn_nb - 1};
  }

  // what the sharded mode's routing needs of a rank's slice: the row-local pass + the (zone, name) -> alias record index
  void prepare_route() {
    alloc_work();
    arm_group_a(1u << IX_ALIAS);
    stage1();
    finish_group_a();
  }
  // a directory shard's tables (gar_shard.h): probes in lbi_*, load balancers, accelerator stubs
  void prepare_directory() {
    alloc_work();
    arm_group_a((1u << IX_LB) | (1u << IX_THOST));
    if (T.o.n_lbi) be.for_each("tokenise_hostnames", T.o.n_lbi, FTokenise{T, W});
    if (T.a.n_accels) be.for_each("digest_accelerators", T.a.n_accels, FDigestAccel{T, W});
    if (T.a.n_lbs) be.for_each("hash_load_balancers", T.a.n_lbs, FLbHash{T, W});
    finish_group_a();
  }

  u32 dport_cap = 0, pair_cap = 0;  // capacities of the two intermediate relations whose size only the device knows
  u64 ops_cap = 0;
  bool tiny_caps = false;  // test hook (environment GAR_TINY_CAPS=1): start every capacity at 1 so that the grow-and-rerun paths run
  int prepare() {
    const u32 n = T.o.n_objects, nacc = T.a.n_accels, nzone = T.a.n_zones, nrec = T.a.n_records, nval = T.a.n_values;
    alloc_work();
    if (!force_radix) {
      arm_group_a((1u << IX_OVN) - 1);
      arm_ovn();
    }
    stage1();
    // stage 2: listen-ports annotation -> desired port lists (count, scan, write).  The total stays on the device: the list
    // buffer has a capacity, a diff that needs more is re-run (run_with)
    be.fill32(W.dport_begin, 0, (size_t)n + 1);
    if (n) be.for_each("listen_ports_count", n, FJsonCount{T, W});
    be.exclusive_scan(W.dport_begin, n + 1);
    be.for_each("gather_header", 1, FGatherHeader{W.dport_begin + n, errflag});
    if (dport_cap < n / 2 + 1024 && !(tiny_caps && dport_cap)) dport_cap = tiny_caps ? 1 : n / 2 + 1024;
    W.dport_cap = dport_cap;
    W.dports = (i32 *)be.out_dports(dport_cap);
    if (n) be.for_each("listen_ports_write", n, FJsonWrite{T, W});

    // stage 3: hash indexes
    u32 *overflow = errflag + FW_IDX_OVERFLOW;
    if (!force_radix) {
      finish_group_a();
      if (nval) be.for_each("value_joins", nval, FValueJoins{T, W});
      finish_ovn();
    } else {  // some bucket was too large for the per-bucket ordering: every index through the stable radix sort
      W.ix_lb = build_index(S_IX_LB, T.a.n_lbs, 1, FRowLb{T, W}, overflow, true);
      W.ix_owner = build_index(S_IX_OWNER, nacc, 1, FRowOwner{T, W}, overflow, true);
      W.ix_thost = build_index(S_IX_THOST, nacc, 1, FRowThost{T, W}, overflow, true);
      W.ix_zone = build_index(S_IX_ZONE, nzone, 1, FRowZone{T}, overflow, true);
      W.ix_val = build_index(S_IX_VAL, nval, 1, FRowVal{T, W}, overflow, true);
      W.ix_alias = build_index(S_IX_ALIAS, nrec, 2, FRowAlias{T, W}, overflow, true);
      W.ix_obj = build_index(S_IX_OBJ, n, 1, FRowObj{T, W}, overflow, true);
      if (nval) be.for_each("value_joins", nval, FValueJoins{T, W});
      W.ix_ovn = build_index(S_IX_OVN, nval, 8, FRowOvn{T, W}, overflow, true);
    }
    return GAR_OK;
  }

  // route53 ensure in relational form over `slots` object slots (rows == nullptr: slot = object row).  The number of
  // (object, hostname) pairs stays on the device: the pair arrays have a capacity (re-run with larger ones if exceeded) and the
  // pair kernel reads its extent from pair_begin[slots].
  u64 n_pairs = 0;  // size of the relation in the last decide (filled from the final read-back; gar_last_counters)
  void r53_relational(u32 slots, const u32 *rows, u32 *st_r53) {
    W.pair_begin = (u32 *)be.ensure(S_PAIR_BEGIN, 4 * (size_t)(slots + 2));
    be.fill32(W.pair_begin, 0, (size_t)slots + 1);
    if (slots) be.for_each_warp("r53_prepare", slots, FR53Prepare{T, W, st_r53, rows});
    be.exclusive_scan(W.pair_begin, slots + 1);
    if (pair_cap < slots + slots / 2 + 1024 && !(tiny_caps && pair_cap)) pair_cap = tiny_caps ? 1 : slots + slots / 2 + 1024;
    W.pair_cap = pair_cap;
    W.pair_obj = (u32 *)be.ensure(S_PAIR_OBJ, 4 * (size_t)(pair_cap + 1));
    W.pair_hn = (gar_str *)be.ensure(S_PAIR_HN, 8 * (size_t)(pair_cap + 1));
    W.pair_code = (u8 *)be.ensure(S_PAIR_CODE, (size_t)pair_cap + 1);
    W.pair_zone = (u32 *)be.ensure(S_PAIR_ZONE, 4 * (size_t)(pair_cap + 1));
    W.pair_rec = (u32 *)be.ensure(S_PAIR_REC, 4 * (size_t)(pair_cap + 1));
    if (slots) {
      be.for_each("r53_fill_pairs", slots, FR53FillPairs{T, W, rows});
      be.for_each_warp_dyn("r53_pairs", W.pair_begin + slots, pair_cap, FR53Pair{T, W});
    }
  }

  // ---- full diff: every object + the orphan sections.  No read-back inside: sizes travel in the flag block (run_with).
  template <class OpsAlloc>
  int decide_all(OpsAlloc ops_alloc) {
    const u32 n = T.o.n_objects, nacc = T.a.n_accels, nrec = T.a.n_records, nval = T.a.n_values;
    // stage 4: evaluate every object once (status + count + staged ops); count the orphan sections
    CountLayout L{n, nacc, nrec, nval};
    u32 *counts = (u32 *)be.ensure(S_COUNTS, 4 * (size_t)(L.total() + 2));
    be.fill32(counts, 0, (size_t)L.total() + 1);
    gar_op *stage_ga = (gar_op *)be.ensure(S_STAGE_GA, sizeof(gar_op) * ((size_t)n * OPS_STAGE_CAP + 1));
    gar_op *stage_r53 = (gar_op *)be.ensure(S_STAGE_R53, sizeof(gar_op) * ((size_t)n * OPS_STAGE_CAP + 1));
    u32 *st_ga = (u32 *)be.out_status_ga(n);
    u32 *st_r53 = (u32 *)be.out_status_r53(n);
    W.acc_claimed = (u8 *)be.ensure(S_ACC_CLAIMED, (size_t)nacc + 4);
    be.fill32((u32 *)W.acc_claimed, 0, ((size_t)nacc + 3) / 4);
    if (n) be.for_each_warp("ga_objects", n, FGaObj{T, W, counts + L.ga_obj(0), stage_ga, st_ga, nullptr});
    r53_relational(n, nullptr, st_r53);
    if (n) be.for_each_warp("r53_objects", n, FR53Obj{T, W, counts + L.r53_obj(0), stage_r53, st_r53, nullptr});
    if (orphan_sweep)
      be.for_each_multi("orphans_count", {nacc, nrec, nval}, FGaOrphan{T, W, L, counts, nullptr, 0}, FR53OrphanAlias{T, W, L, counts, nullptr, 0},
                        FR53OrphanValue{T, W, L, counts, nullptr, 0});
    be.exclusive_scan(counts, L.total() + 1);
    be.for_each("gather_section_begins", 6, FGatherFinal{counts, {0, L.ga_orph(0), L.r53_obj(0), L.base0(), L.total()}, W.pair_begin + n, errflag});

    // stage 5: move ops to their final, canonical positions (writes beyond the buffer's capacity are dropped: the diff is
    // re-run with a larger buffer)
    const u64 est = tiny_caps ? 1 : (u64)n + nacc / 8 + 1024;
    if (ops_cap < est) ops_cap = est;
    gar_op *ops = (gar_op *)ops_alloc(ops_cap);
    const u32 cap = ops_cap > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (u32)ops_cap;
    if (n) be.for_each_warp("ga_objects_compact", n, FCompactOps{T, W, counts + L.ga_obj(0), stage_ga, ops, GAR_CTRL_GA, nullptr, cap});
    if (n) be.for_each_warp("r53_objects_compact", n, FCompactOps{T, W, counts + L.r53_obj(0), stage_r53, ops, GAR_CTRL_R53, nullptr, cap});
    if (orphan_sweep)
      be.for_each_multi("orphans_emit", {nacc, nrec, nval}, FGaOrphan{T, W, L, counts, ops, cap}, FR53OrphanAlias{T, W, L, counts, ops, cap},
                        FR53OrphanValue{T, W, L, counts, ops, cap});
    W.acc_claimed = nullptr;  // other decide flavours (incremental, bindings) do not maintain it
    return GAR_OK;
  }

  // ---- incremental diff: `m` object rows + `nd` deleted keys (device arrays).  counts layout:
  // [GA rows: m][GA deleted keys: nd][R53 rows: m][R53 deleted keys: nd][total]
  template <class OpsAlloc>
  int decide_keys(const u32 *rows, u32 m, DelKeys D, u32 nd, OpsAlloc ops_alloc) {
    const u32 total = 2 * m + 2 * nd;
    u32 *counts = (u32 *)be.ensure(S_COUNTS, 4 * (size_t)(total + 2));
    be.fill32(counts, 0, (size_t)total + 1);
    u32 *c_ga = counts, *c_gad = counts + m, *c_r53 = counts + m + nd, *c_r53d = counts + 2 * m + nd;
    gar_op *stage_ga = (gar_op *)be.ensure(S_STAGE_GA, sizeof(gar_op) * ((size_t)m * OPS_STAGE_CAP + 1));
    gar_op *stage_r53 = (gar_op *)be.ensure(S_STAGE_R53, sizeof(gar_op) * ((size_t)m * OPS_STAGE_CAP + 1));
    u32 *st_ga = (u32 *)be.out_status_ga(m);
    u32 *st_r53 = (u32 *)be.out_status_r53(m);
    u32 *derived_out = (u32 *)be.out_derived_keys(m);
    if (m) {
      be.for_each("gather_derived", m, FGatherDerived{W.derived, rows, derived_out});
      be.for_each_warp("ga_objects", m, FGaObj{T, W, c_ga, stage_ga, st_ga, rows});
    }
    if (nd) be.for_each("ga_deleted_keys_count", nd, FDelKeyGa{T, W, D, c_gad, nullptr, 0});
    r53_relational(m, rows, st_r53);
    if (m) be.for_each_warp("r53_objects", m, FR53Obj{T, W, c_r53, stage_r53, st_r53, rows});
    if (nd) be.for_each("r53_deleted_keys_count", nd, FDelKeyR53{T, W, D, c_r53d, nullptr, 0});
    be.exclusive_scan(counts, total + 1);
    be.for_each("gather_section_begins", 6, FGatherFinal{counts, {0, m, m + nd, 2 * m + nd, total}, W.pair_begin + m, errflag});
    const u64 est = tiny_caps ? 1 : 2 * (u64)m + 4 * (u64)nd + 256;
    if (ops_cap < est) ops_cap = est;
    gar_op *ops = (gar_op *)ops_alloc(ops_cap);
    const u32 cap = ops_cap > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (u32)ops_cap;
    if (m) be.for_each_warp("ga_objects_compact", m, FCompactOps{T, W, c_ga, stage_ga, ops, GAR_CTRL_GA, rows, cap});
    if (nd) be.for_each("ga_deleted_keys_emit", nd, FDelKeyGa{T, W, D, c_gad, ops, cap});
    if (m) be.for_each_warp("r53_objects_compact", m, FCompactOps{T, W, c_r53, stage_r53, ops, GAR_CTRL_R53, rows, cap});
    if (nd) be.for_each("r53_deleted_keys_emit", nd, FDelKeyR53{T, W, D, c_r53d, ops, cap});
    return GAR_OK;
  }

  // ---- EndpointGroupBinding set-diff over `nb` bindings (device pointers in `b`)
  template <class OpsAlloc>
  int decide_bindings(const gar_bindings &b, OpsAlloc ops_alloc) {
    u32 *overflow = errflag + FW_IDX_OVERFLOW;
    const u32 nb = b.n_bindings;
    DevBindings DB{b, build_index(S_IX_EG, b.n_known_egs, 1, FRowKnownEg{b}, overflow, force_radix)};
    u32 *counts = (u32 *)be.ensure(S_COUNTS, 4 * (size_t)(nb + 2));
    be.fill32(counts, 0, (size_t)nb + 1);
    u32 *st = (u32 *)be.out_status_ga(nb);
    if (nb) be.for_each("egb_count", nb, FEgb{T, W, DB, counts, nullptr, nullptr, 0});
    be.exclusive_scan(counts, nb + 1);
    be.for_each("gather_section_begins", 6, FGatherFinal{counts, {0, nb, nb, nb, nb}, nullptr, errflag});
    const u64 est = tiny_caps ? 1 : 4 * (u64)nb + 256;
    if (ops_cap < est) ops_cap = est;
    gar_op *ops = (gar_op *)ops_alloc(ops_cap);
    const u32 cap = ops_cap > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (u32)ops_cap;
    if (nb) be.for_each("egb_emit", nb, FEgb{T, W, DB, counts, ops, st, cap});
    return GAR_OK;
  }

  // prepare (once per snapshot) + one of the decide flavours, then the ONE read-back of the diff: the flag block with the
  // section sizes and everything that may force another attempt — a hash bucket too large for the per-bucket ordering
  // (-> stable radix build), or an intermediate relation larger than its buffer (-> larger buffer).  Retries are rare:
  // capacities only grow, so a snapshot shape settles after its first diff.
  // `replayable`: the launch sequence of this flavour depends only on the snapshot and the capacities, so the backend may record
  // it once and replay it (a CUDA graph): the full diff.  Incremental / binding diffs take new host inputs every time.
  template <class DecideF>
  int run_with(DiffCounts *dc, bool full, DecideF decide) {
    for (int attempt = 0; attempt < 8; attempt++) {
      u64 sig = 0;
      if (full) {
        sig = hmix(hmix(prepared ? 1 : 2, force_radix ? 3 : 4), hmix(hmix(dport_cap, pair_cap), ops_cap));
        sig = hmix(sig, hmix(orphan_sweep ? 5 : 6, tiny_caps ? 7 : 8)) | 1;
      }
      const int g = full ? be.graph_begin(sig) : 0;
      int rc = GAR_OK;
      if (g != 2) {
        if (!prepared) rc = prepare();
        if (rc == GAR_OK) rc = decide();
      }
      prepared = true;
      if (full) be.graph_end();
      if (rc != GAR_OK) return rc;
      u32 fl[FW_WORDS];
      be.download(fl, errflag, sizeof(fl));
      if (fl[FW_BAD_KEYS]) return GAR_E_INVALID;
      if (fl[FW_IDX_OVERFLOW] && !force_radix) {
        force_radix = true;
        prepared = false;
        continue;
      }
      if (fl[FW_NDPORTS] > dport_cap) {
        dport_cap = fl[FW_NDPORTS] + fl[FW_NDPORTS] / 8 + 16;
        prepared = false;
        continue;
      }
      if (fl[FW_NPAIRS] > pair_cap) {
        pair_cap = fl[FW_NPAIRS] + fl[FW_NPAIRS] / 8 + 16;
        continue;
      }
      const u64 nops = fl[FW_SEC0 + 4];
      if (nops > ops_cap) {
        ops_cap = nops + nops / 8 + 16;
        continue;
      }
      n_dports = fl[FW_NDPORTS];
      n_pairs = fl[FW_NPAIRS];
      for (int k = 0; k < 5; k++) dc->section_begin[k] = fl[FW_SEC0 + k];
      dc->n_ops = nops;
      dc->n_dports = full ? n_dports : 0;
      // an EMPTY object table with owned resources left: an unsynced informer looks exactly like this, and the orphan sections
      // would delete everything the cluster owns.  (A shard that happens to home no object is fine: the cluster is not empty.)
      if (full && T.o.n_objects == 0 && !sharded && !allow_empty_cache && nops != 0) return GAR_REFUSE_EMPTY_CACHE;
      return GAR_OK;
    }
    return GAR_E_STATE;
  }
  template <class OpsAlloc>
  int run(DiffCounts *dc, OpsAlloc ops_alloc) {
    return run_with(dc, true, [&] { return decide_all(ops_alloc); });
  }
  template <class OpsAlloc>
  int run_keys(const u32 *rows, u32 m, DelKeys D, u32 nd, DiffCounts *dc, OpsAlloc ops_alloc) {
    return run_with(dc, false, [&] { return decide_keys(rows, m, D, nd, ops_alloc); });
  }
  template <class OpsAlloc>
  int run_bindings(const gar_bindings &b, DiffCounts *dc, OpsAlloc ops_alloc) {
    return run_with(dc, false, [&] { return decide_bindings(b, ops_alloc); });
  }
};
