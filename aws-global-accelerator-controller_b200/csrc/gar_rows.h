// gar_rows.h — per-row decision logic of the diff engine (one call = one table row).
//
// Each function states the reference code it stands for (paths relative to the reference root).
// Everything here is GAR_HD: nvcc compiles it into the sm_100a kernels of libgarecon.so; tests/hostsim
// compiles the same text with g++ for CPU-side debugging of the device logic.
#pragma once

#include "gar_common.h"
#include "gar_json.h"

// ------------------------------------------------------------------ tables + work areas (device pointers)

struct DevTables {
  gar_objects o;
  gar_actual a;
  const u8 *cluster;  // --cluster-name, GAR_SLAB_PAD padded
  u32 cluster_len;
};

// internal per-object bits stored above the public GAR_DV_* byte in Work.derived (masked off before export)
enum {
  OBJ_HAS_NAME_ANN = 1u << 8,
  OBJ_HAS_TAGS_ANN = 1u << 9,
  OBJ_KEY_BAD = 1u << 10,  // ns/name are not laid out as "ns/name" (layout rule violated; engine reports GAR_E_INVALID)
};

// per-accelerator bits (from its tag list)
enum {
  ACC_MINE = 1u << 0,        // managed tag == "true" and cluster tag == --cluster-name (missing tag reads as "")
  ACC_OWNER_KEYED = 1u << 1, // owner tag is "service/<rest>" or "ingress/<rest>": can match an object key
  ACC_OWNER_INGRESS = 1u << 2,
  ACC_OWNER_3PART = 1u << 3, // <rest> contains exactly one '/': a key the controller could have written
  ACC_HAS_MANAGED = 1u << 4, ACC_HAS_OWNER = 1u << 5, ACC_HAS_THOST = 1u << 6,
};

// r53_mode: how the route53 decisions of an object are evaluated
enum {
  R53_MODE_DONE = 0,   // status final after r53_prepare (ignored / early status), no ops
  R53_MODE_PAIRS = 1,  // one lbIngress with a usable accelerator: hostnames are evaluated as (object, hostname) pairs
  R53_MODE_OBJECT = 2, // everything else (cleanup, several lbIngress): the per-object routine r53_reconcile
};
enum { PAIR_IN_SYNC = 0, PAIR_CREATE = 1, PAIR_UPSERT = 2, PAIR_NO_ZONE = 3,
       PAIR_REPEAT = 4 };  // the same hostname string earlier in the annotation: visited a moment ago with the same accelerator -> nothing to do
#define VALNAME_HAS_BACKSLASH (1u << 30)  // ix_val entry a1 bit: the record name contains a backslash (possible \052 escape)

// per-value-row class: is this ResourceRecord value an owner value of this cluster?
enum { VAL_NOT_OWNER = 0, VAL_OWNER_SERVICE = 1, VAL_OWNER_INGRESS = 2, VAL_OWNER_3PART = 4 };

// Everything the Global Accelerator decisions read about one accelerator besides its strings, gathered into ONE
// 64-byte record by the streaming digest pass: the probe side then pays one DRAM burst instead of a dozen scattered
// column reads (acc_enabled, acc_name, acc_lis_begin, lis_proto, lis_pr_begin, pr_from, lis_eg_begin, eg_ep_begin, ep_id ...).
struct alignas(64) AccDigest {
  u32 flags;     // ACC_* | ACCD_*
  u32 lis;       // first listener row (valid if >= 1 listener)
  u32 eg;        // first endpoint-group row of that listener (valid if >= 1)
  u32 pr_begin;  // port ranges of that listener
  u32 ep_begin;  // endpoint descriptions of that endpoint group
  u16 n_ports, n_eps;
  i32 port0, port1;  // the first two FromPorts inline
  gar_str name;       // Accelerator.Name
  gar_str thost;      // target-hostname tag value
  gar_str owner_key;  // owner tag value minus "service/" | "ingress/"
  gar_str ep0;        // first EndpointDescription.EndpointId
};
enum {
  ACCD_ENABLED = 1u << 8,
  ACCD_MANAGED_TRUE = 1u << 9,     // managed tag value == "true"
  ACCD_LIS_NONE = 1u << 10, ACCD_LIS_MANY = 1u << 11,
  ACCD_LIS_UDP = 1u << 12,
  ACCD_EG_NONE = 1u << 13, ACCD_EG_MANY = 1u << 14,
};
struct alignas(16) ValLink {  // per owner value row: first alias A record under the same (zone, name)
  u32 alias_row, pad;
  gar_str alias_dns;
};

// the hash indexes, in build order (group A is built together in one pass, IX_OVN after the per-value joins)
enum IxId { IX_LB, IX_OWNER, IX_THOST, IX_ZONE, IX_VAL, IX_ALIAS, IX_OBJ, IX_OVN, IX_N };
// Bucket histogram hook of the one-pass index build: the row-local passes that PRODUCE a key hash also count its bucket
// (cnt == nullptr: that index is not being built by the fast path).
struct IxHist {
  u32 *cnt;  // [nbuckets] zeroed before the row passes
  u32 mask;
};
#if defined(__CUDA_ARCH__)
#define GAR_HIST_ADD(p) atomicAdd((p), 1u)
#else
#define GAR_HIST_ADD(p) (++*(p))
#endif
GAR_HD void ix_count(const IxHist &h, u64 key_hash) {
  if (h.cnt) GAR_HIST_ADD(&h.cnt[(u32)key_hash & h.mask]);
}

struct Work {
  IxHist hist[IX_N];
  u64 *lb_hash;    // [n_lbs] key_hash_lb(region, name), stored by the LB histogram pass for the placement pass
  u8 *rec_flags;   // [n_records] bit 0: the record name contains a backslash (possible \\052 escape)
  u32 pair_cap;    // capacity of the pair_* arrays (a diff whose pair count exceeds it is re-run with larger arrays)
  u32 dport_cap;   // capacity of dports
  // objects
  u32 *derived;        // [n] GAR_DV_* | OBJ_*
  u64 *okey_hash;      // [n] key_hash_kinded(kind, "ns/name"): probes ix_owner / ix_val, builds ix_obj
  gar_str *ann_r53;    // [n] value of the route53-hostname annotation
  gar_str *ann_name;   // [n] value of global-accelerator-name
  gar_str *ann_tags;   // [n] value of global-accelerator-tags
  gar_str *ann_listen; // [n] value of alb.ingress.kubernetes.io/listen-ports
  u32 *dport_begin;    // [n+1] counts, then exclusive scan
  i32 *dports;
  // lbIngress rows
  u8 *tok_code;
  gar_str *tok_name, *tok_region;
  // accelerators
  u32 *acc_flags;
  gar_str *acc_owner_key;  // owner tag value minus the "service/" | "ingress/" prefix (refs into actual slab)
  gar_str *acc_owner;      // full owner tag value ("" if missing)
  gar_str *acc_thost;      // target-hostname tag value ("" if missing)
  gar_str *acc_managed;    // managed tag value
  AccDigest *acc_digest;   // [n_accels]
  u64 *acc_owner_hash;     // key_hash_kinded(kind, owner key) for ACC_OWNER_KEYED rows
  u64 *acc_thost_hash;     // gar_hash(target hostname)
  // route53 expansion
  u32 *rec_zone;  // [n_records]
  u64 *rec_name_hash;  // [n_records] gar_hash(record name): every (zone, name) key is derived from it
  u32 *val_rec;   // [n_values]
  u8 *val_cls;    // [n_values] VAL_*
  gar_str *val_key;  // [n_values] "<ns>/<name>" part of an owner value
  u64 *val_key_hash; // [n_values] key_hash_kinded(kind, val_key) for owner values
  u8 *val_orphan;    // [n_values] 1 = owner value of this cluster whose object is not in the cache
  ValLink *val_link;      // [n_values] owner values: first alias record of type A under the same (zone, name) + its DNSName
  // sharded mode (gar_shard.h): rows >= acc_guest_from are guest copies that answer by-target-hostname lookups only;
  // the rows below it are this shard's own accelerators (owner-keyed lookups, orphan detection).  Unsharded: 0xFFFFFFFF
  // and every row serves both.
  u32 acc_guest_from;
  u32 sharded;
  u8 *acc_claimed;  // [n_accels] written by ga_reconcile (full diff only; nullptr otherwise), read by ga_orphan
  // route53 ensure, relational form (objects with exactly one lbIngress)
  u8 *r53_mode;        // [n] R53_MODE_*
  u32 *r53_acc;        // [n] the accelerator found by target hostname
  gar_str *r53_acc_dns;// [n] its DnsName
  u32 *pair_begin;     // [n+1] (object, hostname) pairs, CSR
  u32 *pair_obj;       // [n_pairs]
  gar_str *pair_hn;    // [n_pairs] the k-th piece of strings.Split(annotation, ",")
  u8 *pair_code;       // [n_pairs] PAIR_*
  u32 *pair_zone;      // [n_pairs]
  u32 *pair_rec;       // [n_pairs]
  // indexes
  HashIdx ix_lb;     // (region, name) -> LB rows
  HashIdx ix_owner;  // (kind, "ns/name") -> accelerators that are ACC_MINE and ACC_OWNER_KEYED
  HashIdx ix_thost;  // target hostname -> accelerators that are ACC_MINE
  HashIdx ix_zone;   // zone name without the trailing dot -> zone rows
  const u64 *zone_len_mask;  // [4] bit L set: some indexed zone name has L bytes (L >= 255 -> bit 255)
  HashIdx ix_val;    // (kind, "ns/name") -> owner value rows of this cluster
  HashIdx ix_alias;  // (zone, record name) -> alias record rows
  HashIdx ix_obj;    // (kind, "ns/name") -> object rows
  HashIdx ix_ovn;    // (zone, record name) -> orphan owner value rows
};

// which accelerators enter the owner / target-hostname indexes (sharded mode: guest rows answer by-hostname lookups only)
GAR_HD bool acc_in_owner_index(const Work &W, u32 a, u32 fl) { return (fl & ACC_MINE) && (fl & ACC_OWNER_KEYED) && a < W.acc_guest_from; }
GAR_HD bool acc_in_thost_index(const Work &W, u32 a, u32 fl) { return (fl & ACC_MINE) != 0 && (!W.sharded || a >= W.acc_guest_from); }

// ------------------------------------------------------------------ key hashes (build and probe sides must agree)

GAR_HD u64 key_hash_kinded(u32 kind, Str nsname) { return hmix(kind + 1, gar_hash(nsname)); }
GAR_HD u64 key_hash_lb(Str region, Str name) { return hmix(gar_hash(region), gar_hash(name)); }
GAR_HD u64 key_hash_zoned_h(u32 zone, u64 name_hash) { return hmix((u64)zone + 0x100, name_hash); }
GAR_HD u64 key_hash_zoned(u32 zone, Str name) { return key_hash_zoned_h(zone, gar_hash(name)); }
GAR_HD u64 key_hash_str(Str s) { return gar_hash(s); }

// the workqueue key "ns/name" of an object row (cache.MetaNamespaceKeyFunc; reconcile.go:47).  Layout rule of
// gar_objects: name starts one byte after ns ends and that byte is '/'.
GAR_HD Str object_key(const DevTables &T, u32 i) {
  gar_str ns = T.o.obj_ns[i], nm = T.o.obj_name[i];
  return Str{T.o.slab + GAR_STR_OFF(ns), GAR_STR_LEN(ns) + 1 + GAR_STR_LEN(nm)};
}
GAR_HD bool object_key_ok(const DevTables &T, u32 i) {
  gar_str ns = T.o.obj_ns[i], nm = T.o.obj_name[i];
  u64 sep = GAR_STR_OFF(ns) + GAR_STR_LEN(ns);
  return GAR_STR_OFF(nm) == sep + 1 && sep < T.o.slab_len && T.o.slab[sep] == '/';
}

// ------------------------------------------------------------------ (a2) annotation-key filter / row classifier
//
// wasLoadBalancerService (globalaccelerator/service.go:18-26, route53/service.go:19-27), wasALBIngress
// (globalaccelerator/ingress.go:19-27), hasManagedAnnotation (controller.go:250-253), hasHostnameAnnotation
// (route53/controller.go:243-246), plus the annotation reads of global_accelerator.go:35-60,214,225,526 and
// listenerForService's protocol (global_accelerator.go:503-515).

#define ANN_PREFIX "aws-global-accelerator-controller.h3poteto.dev/"

GAR_HD bool proto_is(Str p, char a, char b, char c) {  // strings.ToLower(p) == "abc" for ASCII a, b, c
  return p.n == 3 && (p.p[0] | 0x20) == a && (p.p[1] | 0x20) == b && (p.p[2] | 0x20) == c;
}

GAR_HD void classify_object(const DevTables &T, const Work &W, u32 i) {
  const gar_objects &o = T.o;
  u32 kind = o.obj_kind[i];
  u32 dv = 0;
  bool has_lbtype = false, has_ingclass = false;
  gar_str r53 = 0, name = 0, tags = 0, listen = 0;
  bool has_listen = false;
  for (u32 k = o.obj_ann_begin[i]; k < o.obj_ann_begin[i + 1]; k++) {
    Str key = mkstr(o.slab, o.ann_key[k]);
    gar_str vref = o.ann_val[k];
    if (HAS_PREFIX_LIT(key, ANN_PREFIX)) {
      Str t = substr(key, sizeof(ANN_PREFIX) - 1, key.n - (u32)(sizeof(ANN_PREFIX) - 1));
      if (STREQ_LIT(t, "global-accelerator-managed")) {
        dv |= GAR_DV_GA_MANAGED;
      } else if (STREQ_LIT(t, "route53-hostname")) {
        dv |= GAR_DV_R53_ANNOTATED;
        r53 = vref;
      } else if (STREQ_LIT(t, "client-ip-preservation")) {
        if (STREQ_LIT(mkstr(o.slab, vref), "true")) dv |= GAR_DV_IP_PRESERVE;
        else dv &= ~(u32)GAR_DV_IP_PRESERVE;
      } else if (STREQ_LIT(t, "global-accelerator-name")) {
        dv |= OBJ_HAS_NAME_ANN;
        name = vref;
      } else if (STREQ_LIT(t, "global-accelerator-tags")) {
        dv |= OBJ_HAS_TAGS_ANN;
        tags = vref;
      } else if (STREQ_LIT(t, "ip-address-type")) {
        Str v = mkstr(o.slab, vref);
        if (STREQ_LIT(v, "ipv4") || STREQ_LIT(v, "IPV4")) dv |= GAR_DV_IPV4;
        else dv &= ~(u32)GAR_DV_IPV4;
      }
    } else if (STREQ_LIT(key, "service.beta.kubernetes.io/aws-load-balancer-type")) {
      has_lbtype = true;
    } else if (STREQ_LIT(key, "kubernetes.io/ingress.class")) {
      has_ingclass = true;
    } else if (STREQ_LIT(key, "alb.ingress.kubernetes.io/listen-ports")) {
      has_listen = true;
      listen = vref;
    }
  }
  if (kind == GAR_KIND_SERVICE) {
    bool lbsvc = o.obj_spec_type[i] == GAR_SVC_LOADBALANCER && (has_lbtype || (o.obj_flags[i] & GAR_OBJ_HAS_LB_CLASS));
    if (lbsvc) dv |= GAR_DV_GA_ELIGIBLE | GAR_DV_R53_ELIGIBLE;
    bool udp = false;  // listenerForService: the last port whose protocol is tcp/udp decides
    for (u32 p = o.obj_port_begin[i]; p < o.obj_port_begin[i + 1]; p++) {
      Str pr = mkstr(o.slab, o.port_proto[p]);
      if (proto_is(pr, 'u', 'd', 'p')) udp = true;
      else if (proto_is(pr, 't', 'c', 'p')) udp = false;
    }
    if (udp) dv |= GAR_DV_PROTO_UDP;
  } else {
    bool alb = has_ingclass;
    if ((o.obj_flags[i] & GAR_OBJ_HAS_INGRESS_CLASS) && STREQ_LIT(mkstr(o.slab, o.obj_ingress_class[i]), "alb")) alb = true;
    if (alb) dv |= GAR_DV_GA_ELIGIBLE;
    dv |= GAR_DV_R53_ELIGIBLE;  // the route53 controller does not filter Ingresses (route53/controller.go:130-148)
    if (has_listen) dv |= GAR_DV_PORTS_FROM_ANN;
  }
  if (!object_key_ok(T, i)) dv |= OBJ_KEY_BAD;
  const u64 okh = (dv & OBJ_KEY_BAD) ? 0 : key_hash_kinded(kind, object_key(T, i));
  W.okey_hash[i] = okh;
  if (!(dv & OBJ_KEY_BAD)) ix_count(W.hist[IX_OBJ], okh);
  W.derived[i] = dv;
  W.ann_r53[i] = r53;
  W.ann_name[i] = name;
  W.ann_tags[i] = tags;
  W.ann_listen[i] = listen;
}

// ------------------------------------------------------------------ (a3) LB hostname tokeniser
//
// DetectCloudProvider (pkg/cloudprovider/provider.go:8-17) followed by GetLBNameFromHostname and its helpers
// (pkg/cloudprovider/aws/load_balancer.go:32-93), as a byte scanner instead of six regexps.

// `^([\\w\\-]+)\\-[\\w]+$`: every byte is \\w or '-', and the last '-' has >= 1 byte on both sides.
// Returns the length of group 1, or 0 when the regexp does not match.  8 bytes per step: byte classes by SWAR
// range tests ([0-9], [A-Z], [a-z], '_', '-'); bytes >= 0x80 are never \\w in RE2.
GAR_HD u32 name_dash_id(Str s) {
  u32 last = GAR_NONE;
  for (u32 i = 0; i < s.n; i += 8) {
    u64 w = load_word(s, i);
    u64 pad = s.n - i < 8 ? ~lowmask(s.n - i) & 0x8080808080808080ull : 0;  // bytes beyond the end count as valid
    if (w & 0x8080808080808080ull) return 0;
    u64 dash = swar_eq_exact(w, '-') & ~pad;
    u64 ok = swar_in_range(w, '0', '9') | swar_in_range(w, 'A', 'Z') | swar_in_range(w, 'a', 'z') | swar_eq_exact(w, '_') | dash | pad;
    if (ok != 0x8080808080808080ull) return 0;
    if (dash) last = i + ((63 - clz64(dash)) >> 3);
  }
  if (last == GAR_NONE || last < 1 || last + 1 >= s.n) return 0;
  return last;
}

// the tokeniser proper: h = the hostname bytes, base = its offset in the slab the name/region refs point into
GAR_HD u8 tokenise_str(Str h, u64 base, gar_str *name_out, gar_str *region_out) {
  u8 code;
  gar_str name = 0, region = 0;
  // label boundaries: the first three dots
  u32 d1 = find_byte(h, 0, '.');
  u32 d2 = d1 < h.n ? find_byte(h, d1 + 1, '.') : h.n;
  u32 d3 = d2 < h.n ? find_byte(h, d2 + 1, '.') : h.n;
  if (d1 >= h.n) {
    code = GAR_TOK_PANIC;  // parts[len(parts)-2] with a single part
  } else if (!(STREQ_LIT(h, "amazonaws.com") || HAS_SUFFIX_LIT(h, ".amazonaws.com"))) {
    code = GAR_TOK_NOT_AWS;
  } else if (HAS_SUFFIX_LIT(h, ".elb.amazonaws.com")) {
    // matchALBHostname: subdomain = label 0, region = label 1 (there are >= 4 labels here)
    Str sub = substr(h, 0, d1);
    region = GAR_STR(base + d1 + 1, d2 - d1 - 1);
    if (HAS_PREFIX_LIT(sub, "internal-")) {
      u32 g = name_dash_id(substr(sub, 9, sub.n - 9));
      if (g) {
        code = GAR_TOK_ALB_INTERNAL;
        name = GAR_STR(base + 9, g);
      } else {
        code = GAR_TOK_ERR_INTERNAL_ALB;
      }
    } else {
      u32 g = name_dash_id(sub);
      if (g) {
        code = GAR_TOK_ALB_PUBLIC;
        name = GAR_STR(base, g);
      } else {
        code = GAR_TOK_ERR_PUBLIC_ALB;
      }
    }
  } else {
    // nlbReg `\.elb\..+\.amazonaws\.com$`: some ".elb." at i with >= 1 byte between it and the final
    // ".amazonaws.com" (14 bytes), none of them '\n'.  The right-most candidate has the smallest middle.
    bool nlb = false;
    if (h.n >= 20) {
      // walk the dots left to right (word-wise search) and keep the right-most ".elb." that starts at or before n - 20
      u32 last = GAR_NONE;
      for (u32 i = d1; i <= h.n - 20; i = find_byte(h, i + 1, '.'))
        if (lit_eq_at(h, i, ".elb.")) last = i;
      if (last != GAR_NONE) nlb = find_byte(substr(h, 0, h.n - 14), last + 5, '\n') >= h.n - 14;
    }
    if (!nlb) {
      code = GAR_TOK_ERR_NOT_ELB;
    } else {
      // matchNLBHostname: subdomain = label 0, region = label 2 (>= 5 labels here)
      u32 g = name_dash_id(substr(h, 0, d1));
      if (g) {
        code = GAR_TOK_NLB;
        name = GAR_STR(base, g);
        region = GAR_STR(base + d2 + 1, d3 - d2 - 1);
      } else {
        code = GAR_TOK_ERR_NLB;
      }
    }
  }
  if (code > GAR_TOK_NLB) {
    name = 0;
    region = 0;
  }
  *name_out = name;
  *region_out = region;
  return code;
}
// h = the bytes of lbi_hostname[row] (in the slab, or staged in shared memory by gar_engine.cu k_tokenise_staged)
GAR_HD void tokenise_hostname_at(const DevTables &T, const Work &W, u32 row, Str h) {
  gar_str name, region;
  u8 code = tokenise_str(h, GAR_STR_OFF(T.o.lbi_hostname[row]), &name, &region);
  W.tok_code[row] = code;
  W.tok_name[row] = name;
  W.tok_region[row] = region;
}
GAR_HD void tokenise_hostname(const DevTables &T, const Work &W, u32 row) { tokenise_hostname_at(T, W, row, mkstr(T.o.slab, T.o.lbi_hostname[row])); }

// ------------------------------------------------------------------ (a5) accelerator tag digest
//
// tagsContainsAllValues builds map[key]value from the tag list (later duplicates win) and reads missing
// keys as "" (global_accelerator.go:559-570).  One pass per accelerator extracts the four system tags.

#define TAG_MANAGED "aws-global-accelerator-controller-managed"
#define TAG_OWNER "aws-global-accelerator-owner"
#define TAG_THOST "aws-global-accelerator-target-hostname"
#define TAG_CLUSTER "aws-global-accelerator-cluster"

GAR_HD u32 count_slashes(Str s) { return count_byte(s, '/'); }

GAR_HD void digest_accelerator(const DevTables &T, const Work &W, u32 a) {
  const gar_actual &A = T.a;
  gar_str managed = 0, owner = 0, thost = 0, cluster = 0;
  u32 fl = 0;
  for (u32 t = A.acc_tag_begin[a]; t < A.acc_tag_begin[a + 1]; t++) {
    Str k = mkstr(A.slab, A.tag_key[t]);
    if (STREQ_LIT(k, TAG_MANAGED)) {
      managed = A.tag_val[t];
      fl |= ACC_HAS_MANAGED;
    } else if (STREQ_LIT(k, TAG_OWNER)) {
      owner = A.tag_val[t];
      fl |= ACC_HAS_OWNER;
    } else if (STREQ_LIT(k, TAG_THOST)) {
      thost = A.tag_val[t];
      fl |= ACC_HAS_THOST;
    } else if (STREQ_LIT(k, TAG_CLUSTER)) {
      cluster = A.tag_val[t];
    }
  }
  Str cl = mkstr(A.slab, cluster);
  if (STREQ_LIT(mkstr(A.slab, managed), "true") && streq(cl, Str{T.cluster, T.cluster_len})) fl |= ACC_MINE;
  Str ow = mkstr(A.slab, owner);
  gar_str key = 0;
  if (HAS_PREFIX_LIT(ow, "service/")) {
    fl |= ACC_OWNER_KEYED;
    key = GAR_STR(GAR_STR_OFF(owner) + 8, ow.n - 8);
  } else if (HAS_PREFIX_LIT(ow, "ingress/")) {
    fl |= ACC_OWNER_KEYED | ACC_OWNER_INGRESS;
    key = GAR_STR(GAR_STR_OFF(owner) + 8, ow.n - 8);
  }
  if ((fl & ACC_OWNER_KEYED) && count_slashes(mkstr(A.slab, key)) == 1) fl |= ACC_OWNER_3PART;
  AccDigest d;
  d.flags = fl | (A.acc_enabled[a] ? ACCD_ENABLED : 0) | (STREQ_LIT(mkstr(A.slab, managed), "true") ? ACCD_MANAGED_TRUE : 0);
  d.lis = d.eg = d.pr_begin = d.ep_begin = 0;
  d.n_ports = d.n_eps = 0;
  d.port0 = d.port1 = 0;
  d.ep0 = 0;
  u32 lb = A.acc_lis_begin[a], le = A.acc_lis_begin[a + 1];
  if (le == lb) d.flags |= ACCD_LIS_NONE;
  else if (le - lb > 1) d.flags |= ACCD_LIS_MANY;
  else {
    d.lis = lb;
    if (A.lis_proto[lb] == GAR_PROTO_UDP) d.flags |= ACCD_LIS_UDP;
    d.pr_begin = A.lis_pr_begin[lb];
    u32 np = A.lis_pr_begin[lb + 1] - d.pr_begin;
    d.n_ports = (u16)(np > 0xFFFF ? 0xFFFF : np);
    if (np > 0) d.port0 = A.pr_from[d.pr_begin];
    if (np > 1) d.port1 = A.pr_from[d.pr_begin + 1];
    u32 eb = A.lis_eg_begin[lb], ee = A.lis_eg_begin[lb + 1];
    if (ee == eb) d.flags |= ACCD_EG_NONE;
    else if (ee - eb > 1) d.flags |= ACCD_EG_MANY;
    else {
      d.eg = eb;
      d.ep_begin = A.eg_ep_begin[eb];
      u32 ne = A.eg_ep_begin[eb + 1] - d.ep_begin;
      d.n_eps = (u16)(ne > 0xFFFF ? 0xFFFF : ne);
      if (ne > 0) d.ep0 = A.ep_id[d.ep_begin];
    }
  }
  d.name = A.acc_name[a];
  d.thost = thost;
  d.owner_key = key;
  W.acc_digest[a] = d;
  const u64 owner_hash = (fl & ACC_OWNER_KEYED) ? key_hash_kinded((fl & ACC_OWNER_INGRESS) ? 1u : 0u, mkstr(A.slab, key)) : 0;
  const u64 thost_hash = (fl & ACC_MINE) ? gar_hash(mkstr(A.slab, thost)) : 0;
  W.acc_owner_hash[a] = owner_hash;
  W.acc_thost_hash[a] = thost_hash;
  if (acc_in_owner_index(W, a, fl)) ix_count(W.hist[IX_OWNER], owner_hash);
  if (acc_in_thost_index(W, a, fl)) ix_count(W.hist[IX_THOST], thost_hash);
  W.acc_flags[a] = fl;
  W.acc_owner_key[a] = key;
  W.acc_owner[a] = owner;
  W.acc_thost[a] = thost;
  W.acc_managed[a] = managed;
}

// ------------------------------------------------------------------ (a9) owner values in Route53
//
// Route53OwnerValue (route53.go:18-20): "heritage=aws-global-accelerator-controller,cluster=<c>,<resource>/<ns>/<name>"
// including the double quotes.  A value can only ever equal an owner value computed for THIS cluster if it has
// that shape, so only such values enter the index, keyed like object keys.

#define R53_HERITAGE "\"heritage=aws-global-accelerator-controller,cluster="

GAR_HD void classify_value(const DevTables &T, const Work &W, u32 v) {
  const gar_actual &A = T.a;
  gar_str ref = A.val_value[v];
  const Str s = mkstr(A.slab, ref);
  u8 cls = VAL_NOT_OWNER;
  gar_str key = 0;
  const u32 hl = (u32)(sizeof(R53_HERITAGE) - 1);
  u32 fixed = hl + T.cluster_len + 1 + 8 + 1;  // heritage + cluster + ',' + "service/" + closing quote
  if (s.n >= fixed && HAS_PREFIX_LIT(s, R53_HERITAGE) && streq(substr(s, hl, T.cluster_len), Str{T.cluster, T.cluster_len}) &&
      s.p[hl + T.cluster_len] == ',' && s.p[s.n - 1] == '"') {
    u32 ro = hl + T.cluster_len + 1;
    Str rest = substr(s, ro, s.n - 1 - ro);
    if (HAS_PREFIX_LIT(rest, "service/")) cls = VAL_OWNER_SERVICE;
    else if (HAS_PREFIX_LIT(rest, "ingress/")) cls = VAL_OWNER_INGRESS;
    if (cls) {
      key = GAR_STR(GAR_STR_OFF(ref) + ro + 8, rest.n - 8);
      if (count_slashes(substr(rest, 8, rest.n - 8)) == 1) cls |= VAL_OWNER_3PART;
    }
  }
  W.val_cls[v] = cls;
  W.val_key[v] = key;
  const u64 vkh = cls ? key_hash_kinded((cls & VAL_OWNER_INGRESS) ? 1u : 0u, substr(s, (u32)(GAR_STR_OFF(key) - GAR_STR_OFF(ref)), (u32)GAR_STR_LEN(key))) : 0;
  W.val_key_hash[v] = vkh;
  if (cls) ix_count(W.hist[IX_VAL], vkh);
}

// ------------------------------------------------------------------ index probes
//
// Entry payloads (IdxEntry.a0/a1/s0/s1), filled by the FEnt* functors of gar_pipeline.h:
//   ix_lb     row=lb    a0=lb_state                 s0=lb_name ref     s1=lb_region ref
//   ix_owner  row=accel a0=acc_flags                s0=owner key ref
//   ix_thost  row=accel                             s0=target-hostname ref  s1=acc_dns ref
//   ix_zone   row=zone                              s0=zone_name ref
//   ix_val    row=value a0=record  a1=zone|kind<<31 s0=owner key ref   s1=record name ref
//   ix_alias  row=record a0=zone   a1=rec_type      s0=record name ref s1=alias dns ref
//   ix_obj    row=object a0=kind                    s0="ns/name" ref
//   ix_ovn    row=value a0=record  a1=zone          s0=record name ref s1=value ref

// GetLoadBalancer (load_balancer.go:13-30) on a client bound to `region` (aws.go:23-25): first row wins
GAR_HD u32 find_lb(const DevTables &T, const Work &W, Str region, Str name, u32 *state) {
  Cursor c = idx_open(W.ix_lb, key_hash_lb(region, name));
  IdxEntry e;
  while (idx_next(W.ix_lb, c, &e))
    if (streq(mkstr(T.a.slab, e.s0), name) && streq(mkstr(T.a.slab, e.s1), region)) {
      *state = e.a0;
      return e.row;
    }
  return GAR_NONE;
}

// ListGlobalAcceleratorByResource (global_accelerator.go:87-110) as a cursor over ix_owner
struct OwnerIter {
  Cursor c;
  Str key;
};
GAR_HD OwnerIter owner_open(const Work &W, u64 key_hash, Str key) { return OwnerIter{idx_open(W.ix_owner, key_hash), key}; }
GAR_HD u32 owner_next(const DevTables &T, const Work &W, u32 kind, OwnerIter &it) {
  IdxEntry e;
  while (idx_next(W.ix_owner, it.c, &e)) {
    if ((((e.a0 & ACC_OWNER_INGRESS) != 0) ? 1u : 0u) != kind) continue;
    if (streq(mkstr(T.a.slab, e.s0), it.key)) return e.row;
  }
  return GAR_NONE;
}

// ListGlobalAcceleratorByHostname (global_accelerator.go:62-85): number of matches (saturating at 2), the first
// match and its DnsName ref
GAR_HD u32 find_by_hostname(const DevTables &T, const Work &W, Str hostname, u32 *first, gar_str *first_dns) {
  Cursor c = idx_open(W.ix_thost, key_hash_str(hostname));
  u32 n = 0;
  *first = GAR_NONE;
  IdxEntry e;
  while (idx_next(W.ix_thost, c, &e)) {
    if (!streq(mkstr(T.a.slab, e.s0), hostname)) continue;
    if (n == 0) {
      *first = e.row;
      *first_dns = e.s1;
    }
    if (++n >= 2) break;
  }
  return n;
}

// GetHostedZone (route53.go:335-358) + parentDomain (:383-386)
// A candidate can only equal a zone name of its own length: zone_len_mask has one bit per length that occurs among the
// indexed zone names (lengths >= 255 share bit 255), so most candidates of the parent walk are rejected without a probe.
GAR_HD bool zone_len_possible(const Work &W, u32 n) {
  u32 b = n < 255 ? n : 255;
  return (W.zone_len_mask[b >> 6] >> (b & 63)) & 1ull;
}
GAR_HD u32 find_hosted_zone(const DevTables &T, const Work &W, Str hostname) {
  Str t = hostname;
  for (;;) {
    if (t.n == 0) return GAR_NONE;
    if (zone_len_possible(W, t.n)) {
      Cursor c = idx_open(W.ix_zone, key_hash_str(t));
      IdxEntry e;
      while (idx_next(W.ix_zone, c, &e)) {
        Str zn = mkstr(T.a.slab, e.s0);
        if (zn.n == t.n + 1 && streq(substr(zn, 0, t.n), t)) return e.row;  // zone.Name == target + "." (index holds dotted names only)
      }
    }
    u32 k = find_byte(t, 0, '.');
    if (k >= t.n) return GAR_NONE;  // single label: parent is ""
    t = substr(t, k + 1, t.n - k - 1);
  }
}

// replaceWildcards(name) == hostname + "."  (route53.go:360-371)
GAR_HD bool record_name_matches(Str name, Str hostname) {
  // first occurrence of \052 in name
  u32 w = GAR_NONE;
  for (u32 k = find_byte(name, 0, '\\'); k + 4 <= name.n; k = find_byte(name, k + 1, '\\'))
    if (name.p[k + 1] == '0' && name.p[k + 2] == '5' && name.p[k + 3] == '2') {
      w = k;
      break;
    }
  if (w == GAR_NONE) return name.n == hostname.n + 1 && name.p[name.n - 1] == '.' && streq(substr(name, 0, hostname.n), hostname);
  // unescaped = name[:w] + "*" + name[w+4:]; compare with hostname + "."
  if (name.n - 3 != hostname.n + 1) return false;
  if (name.p[name.n - 1] != '.') return false;
  if (w >= hostname.n || hostname.p[w] != '*') return false;
  if (!streq(substr(name, 0, w), substr(hostname, 0, w))) return false;
  u32 tail = hostname.n - w - 1;  // bytes of hostname after '*'
  return streq(substr(name, w + 4, tail), substr(hostname, w + 1, tail));
}

// ------------------------------------------------------------------ warp-uniform probes
//
// The lookups above, written so that ALL lanes of a warp call them together (lanes without work pass
// active = false).  Every loop — hashing the key, walking the bucket, comparing key bytes — advances under one
// GAR_ANY vote per step, so the 32 lanes issue their loads in the same instruction (32 misses in flight per
// warp instead of one after another) and re-converge at every step.  Only valid inside for_each_warp kernels.

GAR_HD Cursor cursor_none() { return Cursor{0, 0, 0}; }
GAR_HD Cursor u_open(const HashIdx &ix, bool active, u64 h) { return active ? idx_open(ix, h) : cursor_none(); }

// One voted bucket step: loads the next entry of the lanes that are still searching.  Returns whether this lane
// got an entry whose tag matches (the caller then compares keys with u_streq, again all lanes together).
GAR_HD bool u_bucket_step(const HashIdx &ix, bool searching, Cursor &c, IdxEntry *e) {
  bool step = searching && c.pos < c.end;
  if (step) {
    *e = load_entry(ix.ent + c.pos++);
    return e->tag == c.tag;
  }
  return false;
}
#define U_BUCKET_LOOP(searching_expr, cur) for (; GAR_ANY((searching_expr) && (cur).pos < (cur).end);)

// first LB row matching (region, name)  (GetLoadBalancer, load_balancer.go:13-30)
GAR_HD u32 u_find_lb(const DevTables &T, const Work &W, bool active, Str region, Str name, u32 *state) {
  u64 h = hmix(u_hash(active, region), u_hash(active, name));
  Cursor c = u_open(W.ix_lb, active, h);
  u32 found = GAR_NONE;
  U_BUCKET_LOOP(found == GAR_NONE, c) {
    IdxEntry e;
    bool hit = u_bucket_step(W.ix_lb, found == GAR_NONE, c, &e);
    bool eq = u_streq(hit, mkstr(T.a.slab, e.s0), name);
    eq = u_streq(eq, mkstr(T.a.slab, e.s1), region);
    if (eq) {
      found = e.row;
      *state = e.a0;
    }
  }
  return found;
}

// next accelerator of the owner key (ListGlobalAcceleratorByResource, global_accelerator.go:87-110); the cursor
// lives in the caller: one call = one accelerator, all lanes together
GAR_HD u32 u_owner_next(const DevTables &T, const Work &W, bool active, u32 kind, Str key, Cursor &c) {
  u32 found = GAR_NONE;
  U_BUCKET_LOOP(active && found == GAR_NONE, c) {
    IdxEntry e;
    bool hit = u_bucket_step(W.ix_owner, active && found == GAR_NONE, c, &e);
    hit = hit && (((e.a0 & ACC_OWNER_INGRESS) != 0) ? 1u : 0u) == kind;
    if (u_streq(hit, mkstr(T.a.slab, e.s0), key)) found = e.row;
  }
  // an accelerator reached through its owner's object cannot be an orphan: the orphan pass skips its cache probe
  if (found != GAR_NONE && W.acc_claimed) W.acc_claimed[found] = 1;
  return found;
}

// accelerators whose target-hostname tag equals `hostname` (ListGlobalAcceleratorByHostname, :62-85):
// count (saturating at 2), first row, its DnsName
GAR_HD u32 u_find_by_hostname(const DevTables &T, const Work &W, bool active, Str hostname, u32 *first, gar_str *first_dns) {
  Cursor c = u_open(W.ix_thost, active, u_hash(active, hostname));
  u32 n = 0;
  *first = GAR_NONE;
  U_BUCKET_LOOP(n < 2, c) {
    IdxEntry e;
    bool hit = u_bucket_step(W.ix_thost, n < 2, c, &e);
    if (u_streq(hit, mkstr(T.a.slab, e.s0), hostname)) {
      if (n == 0) {
        *first = e.row;
        *first_dns = e.s1;
      }
      n++;
    }
  }
  return n;
}

// GetHostedZone (route53.go:335-358): one voted round per candidate suffix
GAR_HD u32 u_find_hosted_zone(const DevTables &T, const Work &W, bool active, Str hostname) {
  Str t = hostname;
  u32 zone = GAR_NONE;
  bool walking = active;
  for (;;) {
    bool round = walking && t.n != 0;
    if (!GAR_ANY(round)) break;
    bool probe = round && zone_len_possible(W, t.n);
    Cursor c = u_open(W.ix_zone, probe, u_hash(probe, t));
    U_BUCKET_LOOP(zone == GAR_NONE, c) {
      IdxEntry e;
      bool hit = u_bucket_step(W.ix_zone, zone == GAR_NONE, c, &e);
      Str zn = mkstr(T.a.slab, e.s0);
      hit = hit && zn.n == t.n + 1;  // zone.Name == target + "." (the index holds dotted names only)
      if (u_streq(hit, substr(zn, 0, hit ? t.n : 0), t)) zone = e.row;
    }
    u32 k = u_find_byte(round && zone == GAR_NONE, t, 0, '.');
    if (round) {
      if (zone != GAR_NONE || k >= t.n) walking = false;  // found, or single label left: parent is ""
      else t = substr(t, k + 1, t.n - k - 1);
    }
  }
  return zone;
}

// first alias record with type A under (zone, name)
GAR_HD u32 u_first_alias_a(const DevTables &T, const Work &W, bool active, u32 zone, Str name, gar_str *alias_dns) {
  Cursor c = u_open(W.ix_alias, active, hmix((u64)zone + 0x100, u_hash(active, name)));
  u32 found = GAR_NONE;
  U_BUCKET_LOOP(found == GAR_NONE, c) {
    IdxEntry e;
    bool hit = u_bucket_step(W.ix_alias, found == GAR_NONE, c, &e);
    hit = hit && e.a0 == zone && e.a1 == GAR_RR_A;
    if (u_streq(hit, mkstr(T.a.slab, e.s0), name)) {
      found = e.row;
      *alias_dns = e.s1;
    }
  }
  return found;
}

// replaceWildcards(name) == hostname + "."  (route53.go:360-371), all lanes together.  Names without a backslash
// (everything but wildcard records) take the voted compare; the \052 case falls back to the scalar routine.
GAR_HD bool u_record_name_matches(bool active, Str name, Str hostname) {
  u32 bs = u_find_byte(active, name, 0, '\\');
  bool plain = active && bs >= name.n;
  bool shape = plain && name.n == hostname.n + 1 && name.p[name.n - 1] == '.';
  bool eq = u_streq(shape, substr(name, 0, shape ? hostname.n : 0), hostname);
  if (active && !plain) eq = record_name_matches(name, hostname);
  return eq;
}

// ------------------------------------------------------------------ op sink (count pass or write pass)

struct OpSink {
  gar_op *out;  // nullptr: count only
  u32 n;
  u32 cap;      // ops beyond cap are counted but not stored (staging slots are small; see FCompactOps)
  GAR_HD void put(u32 head, u32 obj, u32 sub, u32 a0, u32 a1, u32 a2) {
    if (out && n < cap) {
      gar_op o;
      o.head = head;
      o.obj = obj;
      o.sub = sub;
      o.a0 = a0;
      o.a1 = a1;
      o.a2 = a2;
      out[n] = o;
    }
    n++;
  }
};

// ------------------------------------------------------------------ (a4)(a7) desired listener vs actual listener

// desired port list of an object: the input list, or the parsed annotation
struct PortList {
  const i32 *p;
  u32 n;
};
GAR_HD PortList desired_ports(const DevTables &T, const Work &W, u32 i) {
  if (W.derived[i] & GAR_DV_PORTS_FROM_ANN) {
    u32 b = W.dport_begin[i], e = W.dport_begin[i + 1];
    if (e > W.dport_cap) b = e = 0;  // more parsed ports than the buffer holds: the diff is re-run with a larger one
    return PortList{W.dports + b, e - b};
  }
  u32 b = T.o.obj_port_begin[i];
  return PortList{T.o.port_number + b, T.o.obj_port_begin[i + 1] - b};
}

// listenerPortChangedFrom{Service,Ingress} (global_accelerator.go:458-492): build count[port] over
// listener FromPorts and desired ports; changed iff some port has count <= 1, i.e. occurs exactly once in
// the concatenation of both lists.
GAR_HD bool ports_changed(PortList l, PortList d) {
  // A port that sits at the same position in both lists occurs at least twice in the concatenation, so it can never be
  // the witness.  Strip the common prefix and the common suffix; only the ports of the two middle parts (usually 0-2
  // of them: one drifted or extra port) have to be counted against the full lists.  Exact for every input; shuffled
  // lists degrade to the quadratic count.
  u32 nmin = l.n < d.n ? l.n : d.n;
  u32 pre = 0;
  while (pre < nmin && l.p[pre] == d.p[pre]) pre++;
  u32 suf = 0;
  while (suf < nmin - pre && l.p[l.n - 1 - suf] == d.p[d.n - 1 - suf]) suf++;
  u32 ml = l.n - pre - suf, md = d.n - pre - suf;  // middle lengths
  for (u32 x = 0; x < ml + md; x++) {
    i32 px = x < ml ? l.p[pre + x] : d.p[pre + (x - ml)];
    u32 cnt = 0;
    for (u32 y = 0; y < l.n && cnt < 2; y++) cnt += (l.p[y] == px);
    for (u32 y = 0; y < d.n && cnt < 2; y++) cnt += (d.p[y] == px);
    if (cnt <= 1) return true;
  }
  return false;
}

// acceleratorName(resource, obj) == *accelerator.Name  (global_accelerator.go:53-60, :417)
GAR_HD bool accel_name_matches(const DevTables &T, const Work &W, u32 i, u32 kind, Str acc_name) {
  if (W.derived[i] & OBJ_HAS_NAME_ANN) {
    Str n = mkstr(T.o.slab, W.ann_name[i]);
    if (n.n != 0) return streq(n, acc_name);
  }
  // resource + "-" + ns + "-" + name
  Str ns = mkstr(T.o.slab, T.o.obj_ns[i]), nm = mkstr(T.o.slab, T.o.obj_name[i]);
  if (acc_name.n != 7 + 1 + ns.n + 1 + nm.n) return false;
  const u64 res = kind == GAR_KIND_SERVICE ? 0x2d65636976726573ull /* "service-" */ : 0x2d73736572676e69ull /* "ingress-" */;
  if (ld64u(acc_name.p) != res) return false;
  if (acc_name.p[8 + ns.n] != '-') return false;
  return streq(substr(acc_name, 8, ns.n), ns) && streq(substr(acc_name, 9 + ns.n, nm.n), nm);
}

// value of tag `key` in the accelerator's tag list: later duplicates win, missing reads as ""
GAR_HD Str actual_tag(const DevTables &T, u32 acc, Str key) {
  Str v{T.a.slab, 0};
  for (u32 t = T.a.acc_tag_begin[acc]; t < T.a.acc_tag_begin[acc + 1]; t++)
    if (streq(mkstr(T.a.slab, T.a.tag_key[t]), key)) v = mkstr(T.a.slab, T.a.tag_val[t]);
  return v;
}

// One piece of the tags annotation: strings.Split(piece, "=") has exactly two parts
struct TagPiece {
  Str key, val;
  bool ok;
};
GAR_HD TagPiece tag_piece(Str piece) {
  u32 eq = find_byte(piece, 0, '=');
  TagPiece t;
  t.ok = eq < piece.n && find_byte(piece, eq + 1, '=') >= piece.n;
  if (t.ok) {
    t.key = substr(piece, 0, eq);
    t.val = substr(piece, eq + 1, piece.n - eq - 1);
  } else {
    t.key = t.val = Str{piece.p, 0};
  }
  return t;
}
// iterate the pieces of strings.Split(annotation, ",")
GAR_HD bool next_piece(Str all, u32 *pos, Str *piece) {
  if (*pos > all.n) return false;
  u32 b = *pos;
  u32 k = find_byte(all, b, ',');
  *piece = substr(all, b, k - b);
  *pos = k + 1;
  return true;
}

// tag half of acceleratorChanged (global_accelerator.go:420-436), scalar
GAR_HD bool accelerator_tags_changed(const DevTables &T, const Work &W, u32 i, u32 kind, u32 acc, Str lb_dns) {
  const gar_actual &A = T.a;
  // targetTags = {managed:"true", owner:resource/ns/name, target-hostname:lb dns} overlaid by the user tags of
  // the annotation (later pieces overwrite earlier ones and the three system keys).
  bool user_managed = false, user_owner = false, user_thost = false;
  if (W.derived[i] & OBJ_HAS_TAGS_ANN) {
    Str tags = mkstr(T.o.slab, W.ann_tags[i]);
    u32 pos = 0;
    Str piece;
    while (next_piece(tags, &pos, &piece)) {
      TagPiece tp = tag_piece(piece);
      if (!tp.ok) continue;
      if (STREQ_LIT(tp.key, TAG_MANAGED)) user_managed = true;
      else if (STREQ_LIT(tp.key, TAG_OWNER)) user_owner = true;
      else if (STREQ_LIT(tp.key, TAG_THOST)) user_thost = true;
      // overridden by a later piece with the same key?
      bool overridden = false;
      u32 pos2 = pos;
      Str piece2;
      while (next_piece(tags, &pos2, &piece2)) {
        TagPiece t2 = tag_piece(piece2);
        if (t2.ok && streq(t2.key, tp.key)) {
          overridden = true;
          break;
        }
      }
      if (overridden) continue;
      if (!streq(actual_tag(T, acc, tp.key), tp.val)) return true;
    }
  }
  u32 fl = W.acc_flags[acc];
  if (!user_managed && !STREQ_LIT(mkstr(A.slab, W.acc_managed[acc]), "true")) return true;
  if (!user_owner) {
    // owner == resource/ns/name
    bool ok = (fl & ACC_OWNER_KEYED) && (((fl & ACC_OWNER_INGRESS) ? 1u : 0u) == kind) && streq(mkstr(A.slab, W.acc_owner_key[acc]), object_key(T, i));
    if (!ok) return true;
  }
  if (!user_thost && !streq(mkstr(A.slab, W.acc_thost[acc]), lb_dns)) return true;
  return false;
}

// CleanupGlobalAccelerator / listRelatedGlobalAccelerator (global_accelerator.go:254-288): the delete op of one accelerator
GAR_HD void put_delete_chain(const DevTables &T, OpSink &s, u32 obj, u32 kind, u32 acc) {
  const gar_actual &A = T.a;
  u32 lb = A.acc_lis_begin[acc], le = A.acc_lis_begin[acc + 1];
  u32 lis = GAR_NONE, eg = GAR_NONE;
  if (le - lb == 1) {
    lis = lb;
    u32 eb = A.lis_eg_begin[lis], ee = A.lis_eg_begin[lis + 1];
    if (ee - eb == 1) eg = eb;
  }
  s.put(GAR_OP_HEAD(GAR_OP_GA_DELETE_CHAIN, GAR_CTRL_GA, obj == GAR_NONE ? 0 : kind), obj, 0, acc, lis, eg);
}

// ------------------------------------------------------------------ (a6)(a7)(a8) Global Accelerator decisions of one object
//
// process{Service,Ingress}CreateOrUpdate (globalaccelerator/service.go:54-126, ingress.go:56-130) with
// EnsureGlobalAcceleratorFor* (global_accelerator.go:112-211) and updateGlobalAcceleratorFor* (:290-410) inlined.

// acceleratorChanged (global_accelerator.go:412-437), all lanes together.  The rare tags-annotation overlay keeps the
// scalar routine (divergent, no votes inside).
GAR_HD bool u_accelerator_changed(const DevTables &T, const Work &W, bool act, u32 i, u32 dv, u32 kind, u32 acc, const AccDigest &d, Str okey, Str lb_dns) {
  const gar_actual &A = T.a;
  bool ch = act && !(d.flags & ACCD_ENABLED);
  // name: the annotation when non-empty, else resource-ns-name
  bool need = act && !ch;
  Str an = need ? mkstr(A.slab, d.name) : Str{A.slab, 0};
  Str ann = (need && (dv & OBJ_HAS_NAME_ANN)) ? mkstr(T.o.slab, W.ann_name[i]) : Str{T.o.slab, 0};
  bool by_ann = need && ann.n != 0;
  bool eq_ann = u_streq(by_ann, ann, an);
  Str ns = need ? mkstr(T.o.slab, T.o.obj_ns[i]) : Str{T.o.slab, 0};
  Str nm = need ? mkstr(T.o.slab, T.o.obj_name[i]) : Str{T.o.slab, 0};
  bool shape = need && !by_ann && an.n == 9 + ns.n + nm.n &&
               ld64u(an.p) == (kind == GAR_KIND_SERVICE ? 0x2d65636976726573ull /* "service-" */ : 0x2d73736572676e69ull /* "ingress-" */) &&
               an.p[8 + ns.n] == '-';
  bool eq_def = u_streq(shape, substr(an, 8, shape ? ns.n : 0), ns);
  eq_def = u_streq(eq_def, substr(an, 9 + ns.n, eq_def ? nm.n : 0), nm);
  if (need && !(by_ann ? eq_ann : eq_def)) ch = true;
  // tags: managed, owner, target-hostname (user tags from the annotation may override them)
  bool tagcheck = act && !ch;
  bool overlay = tagcheck && (dv & OBJ_HAS_TAGS_ANN);
  if (overlay) ch = accelerator_tags_changed(T, W, i, kind, acc, lb_dns);
  bool sys = tagcheck && !overlay;
  u32 fl = d.flags;
  if (sys && !(fl & ACCD_MANAGED_TRUE)) ch = true;
  // the owner tag equals resource/ns/name: guaranteed by the index probe that produced `acc` (kind + key compared there)
  bool th = sys && !ch;
  bool th_eq = u_streq(th, th ? mkstr(A.slab, d.thost) : Str{A.slab, 0}, lb_dns);
  if (th && !th_eq) ch = true;
  return ch;
}

// ---- self-observation (include/garecon.h): what an object's own earlier ops mean for its later lbIngress iterations.
// Everything here is scalar (no votes): objects with a second load balancer that reaches the update stage are rare.

// What the object's user tags do, once written, to the tags ListGlobalAcceleratorByResource filters on (global_accelerator.go:99-103)
// and to the target-hostname tag (createAccelerator :654-675 / updateAccelerator :720-735 append them after the system tags; a tag
// list reads "later duplicate wins", :560-563).
GAR_HD void user_tag_effects(const DevTables &T, const Work &W, u32 i, u32 kind, Str okey, bool *keep_visible, bool *user_thost) {
  *keep_visible = true;
  *user_thost = false;
  if (!(W.derived[i] & OBJ_HAS_TAGS_ANN)) return;
  Str tags = mkstr(T.o.slab, W.ann_tags[i]);
  bool m_ok = true, o_ok = true, c_ok = true;  // verdict of the LAST ok piece of each key
  u32 pos = 0;
  Str piece;
  while (next_piece(tags, &pos, &piece)) {
    TagPiece tp = tag_piece(piece);
    if (!tp.ok) continue;
    if (STREQ_LIT(tp.key, TAG_MANAGED)) m_ok = STREQ_LIT(tp.val, "true");
    else if (STREQ_LIT(tp.key, TAG_OWNER))
      o_ok = tp.val.n == 8 + okey.n && (kind == GAR_KIND_SERVICE ? lit_eq_at(tp.val, 0, "service/") : lit_eq_at(tp.val, 0, "ingress/")) &&
             streq(substr(tp.val, 8, okey.n), okey);
    else if (STREQ_LIT(tp.key, TAG_CLUSTER)) c_ok = streq(tp.val, Str{T.cluster, T.cluster_len});
    else if (STREQ_LIT(tp.key, TAG_THOST)) *user_thost = true;
  }
  *keep_visible = m_ok && o_ok && c_ok;
}
// endpointContainsLB (:494-501) on the snapshot's endpoint group of a digested accelerator
GAR_HD bool eg_contains(const DevTables &T, const AccDigest &d, Str lb_arn) {
  u32 nep = d.n_eps == 0xFFFF ? T.a.eg_ep_begin[d.eg + 1] - d.ep_begin : d.n_eps;
  for (u32 x = 0; x < nep; x++)
    if (streq(mkstr(T.a.slab, x == 0 ? d.ep0 : T.a.ep_id[d.ep_begin + x]), lb_arn)) return true;
  return false;
}
// A later iteration (the object already went through the update/create stage with load balancer prev_lb):
//   * its accelerators satisfy acceleratorChanged for prev_lb, have one desired listener and one endpoint group;
//   * an endpoint group that was created or replaced holds exactly [prev_lb] (updateEndpointGroup replaces, :987-1002),
//     an untouched one the snapshot's list;
//   * the accelerator of an earlier GA_CREATE_CHAIN is listed as GAR_PENDING — unless the user tags overwrite a tag the
//     list call filters on: then nothing the object wrote is listed and the reference creates again.
GAR_HD void ga_later_step(const DevTables &T, const Work &W, u32 i, u32 kind, Str okey, u64 okh, u32 jb, u32 j, u32 lb, u32 prev_lb, bool pending, OpSink &s, u32 *ev);

// Written warp-synchronously: every lane of the warp runs the same outer loops (lbIngress index, accelerator of the
// owner) and the same probe / compare steps under GAR_ANY votes, carrying its own predicates; nothing returns from
// inside a loop.  `valid` is false for padding lanes beyond the last object.
GAR_HD u32 ga_reconcile(const DevTables &T, const Work &W, u32 i, bool valid, OpSink &s) {
  const gar_objects &o = T.o;
  const gar_actual &A = T.a;
  u32 result = GAR_STATUS(GAR_ST_IGNORED, 0, 0);
  u32 dv = 0, kind = 0, jb = 0, nj = 0;
  Str okey{T.o.slab, 0};
  u64 okh = 0;
  bool ensure = false;
  if (valid) {
    dv = W.derived[i];
    if (dv & GAR_DV_GA_ELIGIBLE) {
      jb = o.obj_lbi_begin[i];
      nj = o.obj_lbi_begin[i + 1] - jb;
      kind = o.obj_kind[i];
      if (nj < 1) {
        result = GAR_STATUS(GAR_ST_SKIP_NO_LB, 0, 0);
      } else {
        okey = object_key(T, i);
        okh = W.okey_hash[i];
        if (!(dv & GAR_DV_GA_MANAGED)) {  // cleanup path (rare): runs divergent, no votes inside
          OwnerIter it = owner_open(W, okh, okey);
          for (u32 acc; (acc = owner_next(T, W, kind, it)) != GAR_NONE;) put_delete_chain(T, s, i, kind, acc);
          result = GAR_STATUS(GAR_ST_OK, 0, GAR_EV_DELETED);
        } else {
          ensure = true;
        }
      }
    }
  }
  u32 ev = 0;
  bool stop = false;
  u32 prev_lb = GAR_NONE;  // load balancer of the previous iteration that reached the update/create stage
  bool pending = false;    // that stage emitted GA_CREATE_CHAIN: later iterations see a GAR_PENDING accelerator
  for (u32 j = 0;; j++) {
    bool act = ensure && !stop && j < nj;
    if (!GAR_ANY(act)) break;
    bool probe = false;
    Str hostname{o.slab, 0}, tregion{o.slab, 0}, tname{o.slab, 0};
    if (act) {
      u32 code = W.tok_code[jb + j];
      if (code == GAR_TOK_PANIC) {
        result = GAR_STATUS(GAR_ST_PANIC, 0, ev);
        stop = true;
      } else if (code == GAR_TOK_NOT_AWS) {
      } else if (code >= GAR_TOK_ERR_NOT_ELB) {
        result = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_NOT_ELB + (code - GAR_TOK_ERR_NOT_ELB), ev);
        stop = true;
      } else {
        probe = true;
        hostname = mkstr(o.slab, o.lbi_hostname[jb + j]);
        tregion = mkstr(o.slab, W.tok_region[jb + j]);
        tname = mkstr(o.slab, W.tok_name[jb + j]);
      }
    }
    // EnsureGlobalAcceleratorFor* (global_accelerator.go:112-211)
    u32 lb_state = 0;
    u32 lb = u_find_lb(T, W, probe, tregion, tname, &lb_state);
    bool have_lb = probe && lb != GAR_NONE;
    Str lb_dns = have_lb ? mkstr(A.slab, A.lb_dns[lb]) : Str{A.slab, 0};
    bool dns_eq = u_streq(have_lb, lb_dns, hostname);
    bool go = false;
    if (probe) {
      if (!have_lb) {
        result = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_LB_NOT_FOUND, ev);
        stop = true;
      } else if (!dns_eq) {
        result = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_LB_DNS_MISMATCH, ev);
        stop = true;
      } else if (lb_state != GAR_LB_ACTIVE) {
        result = GAR_STATUS(GAR_ST_REQUEUE_30S, 0, ev);
        stop = true;
      } else {
        go = true;
      }
    }
    // the first iteration that gets here evaluates the snapshot (all lanes together); later ones (rare) evaluate what the
    // object's own earlier ops left behind, scalar
    const bool later = go && prev_lb != GAR_NONE;
    if (later) ga_later_step(T, W, i, kind, okey, okh, jb, j, lb, prev_lb, pending, s, &ev);
    go = go && !later;
    Cursor oc = u_open(W.ix_owner, go, okh);
    Str lb_arn = go ? mkstr(A.slab, A.lb_arn[lb]) : Str{A.slab, 0};
    u32 nacc = 0;
    for (;;) {  // accelerators of the owner, in ListAccelerators order
      u32 acc = u_owner_next(T, W, go && !stop, kind, okey, oc);
      bool a = acc != GAR_NONE;
      if (!GAR_ANY(a)) break;
      if (a) nacc++;
      AccDigest d;
      d.flags = 0;
      if (a) d = W.acc_digest[acc];
      // updateGlobalAcceleratorFor{Service,Ingress} (:290-410)
      if (u_accelerator_changed(T, W, a, i, dv, kind, acc, d, okey, lb_dns)) s.put(GAR_OP_HEAD(GAR_OP_GA_UPDATE_ACCEL, GAR_CTRL_GA, kind), i, j, acc, lb, GAR_NONE);
      u32 eg = GAR_NONE;
      if (a) {
        if (d.flags & ACCD_LIS_MANY) {
          result = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_TOO_MANY_LISTENERS, ev);
          stop = true;
        } else if (d.flags & ACCD_LIS_NONE) {
          // the listener is created from the desired state, so neither change predicate fires on it; it has no
          // endpoint group yet, and the one created for it contains the LB (:298-345)
          s.put(GAR_OP_HEAD(GAR_OP_GA_CREATE_LISTENER, GAR_CTRL_GA, kind), i, j, acc, GAR_NONE, GAR_NONE);
          s.put(GAR_OP_HEAD(GAR_OP_GA_CREATE_EG, GAR_CTRL_GA, kind), i, j, acc, GAR_NONE, lb);
        } else {
          u32 lis = d.lis;
          bool want_udp = kind == GAR_KIND_SERVICE && (dv & GAR_DV_PROTO_UDP);
          bool changed = ((d.flags & ACCD_LIS_UDP) != 0) != want_udp;  // :439-456
          if (!changed) {
            PortList want = desired_ports(T, W, i);
            // the common shapes compare against the inline ports; anything else reads the port-range rows
            if (d.n_ports <= 2 && want.n == d.n_ports && (d.n_ports < 1 || want.p[0] == d.port0) && (d.n_ports < 2 || (want.p[1] == d.port1 && d.port0 != d.port1))) changed = false;
            else changed = ports_changed(PortList{A.pr_from + d.pr_begin, d.n_ports == 0xFFFF ? A.lis_pr_begin[lis + 1] - d.pr_begin : d.n_ports}, want);
          }
          if (changed) s.put(GAR_OP_HEAD(GAR_OP_GA_UPDATE_LISTENER, GAR_CTRL_GA, kind), i, j, acc, lis, GAR_NONE);
          if (d.flags & ACCD_EG_MANY) {
            result = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_TOO_MANY_EGS, ev);
            stop = true;
          } else if (d.flags & ACCD_EG_NONE) {
            s.put(GAR_OP_HEAD(GAR_OP_GA_CREATE_EG, GAR_CTRL_GA, kind), i, j, acc, lis, lb);
          } else {
            eg = d.eg;
          }
        }
      }
      // endpointContainsLB (:494-501): one voted step per endpoint description (the first id comes from the digest)
      bool contains = false;
      u32 nep = eg != GAR_NONE ? (d.n_eps == 0xFFFF ? A.eg_ep_begin[eg + 1] - d.ep_begin : d.n_eps) : 0;
      for (u32 x = 0;; x++) {
        bool more = !contains && x < nep;
        if (!GAR_ANY(more)) break;
        gar_str id = more ? (x == 0 ? d.ep0 : A.ep_id[d.ep_begin + x]) : 0;
        if (u_streq(more, mkstr(A.slab, id), lb_arn)) contains = true;
      }
      if (eg != GAR_NONE && !contains) s.put(GAR_OP_HEAD(GAR_OP_GA_UPDATE_EG, GAR_CTRL_GA, kind), i, j, acc, eg, lb);
    }
    if (go && !stop && nacc == 0) {
      s.put(GAR_OP_HEAD(GAR_OP_GA_CREATE_CHAIN, GAR_CTRL_GA, kind), i, j, lb, GAR_NONE, GAR_NONE);
      ev |= GAR_EV_CREATED;
      pending = true;
    }
    if ((go || later) && !stop) prev_lb = lb;
  }
  if (ensure && !stop) result = GAR_STATUS(GAR_ST_OK, 0, ev);
  return result;
}

GAR_HD void ga_later_step(const DevTables &T, const Work &W, u32 i, u32 kind, Str okey, u64 okh, u32 jb, u32 j, u32 lb, u32 prev_lb, bool pending, OpSink &s, u32 *ev) {
  const gar_actual &A = T.a;
  bool keep_visible, user_thost;
  user_tag_effects(T, W, i, kind, okey, &keep_visible, &user_thost);
  if (!keep_visible) {  // nothing this object wrote is listed any more: the list is empty again
    s.put(GAR_OP_HEAD(GAR_OP_GA_CREATE_CHAIN, GAR_CTRL_GA, kind), i, j, lb, GAR_NONE, GAR_NONE);
    *ev |= GAR_EV_CREATED;
    return;
  }
  Str lb_arn = mkstr(A.slab, A.lb_arn[lb]);
  const bool dns_differs = !user_thost && !streq(mkstr(A.slab, A.lb_dns[lb]), mkstr(A.slab, A.lb_dns[prev_lb]));
  const bool arn_differs = !streq(lb_arn, mkstr(A.slab, A.lb_arn[prev_lb]));
  if (pending) {
    if (dns_differs) s.put(GAR_OP_HEAD(GAR_OP_GA_UPDATE_ACCEL, GAR_CTRL_GA, kind), i, j, GAR_PENDING, lb, GAR_NONE);
    if (arn_differs) s.put(GAR_OP_HEAD(GAR_OP_GA_UPDATE_EG, GAR_CTRL_GA, kind), i, j, GAR_PENDING, GAR_PENDING, lb);
  }
  OwnerIter it = owner_open(W, okh, okey);
  for (u32 acc; (acc = owner_next(T, W, kind, it)) != GAR_NONE;) {
    if (dns_differs) s.put(GAR_OP_HEAD(GAR_OP_GA_UPDATE_ACCEL, GAR_CTRL_GA, kind), i, j, acc, lb, GAR_NONE);
    const AccDigest d = W.acc_digest[acc];
    // (more than one listener / endpoint group ended the object at its first iteration)
    const bool created = (d.flags & (ACCD_LIS_NONE | ACCD_EG_NONE)) != 0;
    // replaced so far <=> created, or some earlier iteration's load balancer was not in the snapshot's endpoint list
    bool replaced = created;
    for (u32 jp = 0; jp < j && !replaced; jp++) {
      if (W.tok_code[jb + jp] > GAR_TOK_NLB) continue;  // DetectCloudProvider error: that iteration was skipped
      u32 st;
      u32 lbp = find_lb(T, W, mkstr(T.o.slab, W.tok_region[jb + jp]), mkstr(T.o.slab, W.tok_name[jb + jp]), &st);
      if (lbp != GAR_NONE && !eg_contains(T, d, mkstr(A.slab, A.lb_arn[lbp]))) replaced = true;
    }
    const bool contains = replaced ? !arn_differs : eg_contains(T, d, lb_arn);
    if (!contains) s.put(GAR_OP_HEAD(GAR_OP_GA_UPDATE_EG, GAR_CTRL_GA, kind), i, j, acc, created ? GAR_PENDING : d.eg, lb);
  }
}

// ------------------------------------------------------------------ (a9)(a10) Route53 decisions of one object
//
// process{Service,Ingress}CreateOrUpdate of the route53 controller (route53/service.go:48-111, ingress.go:40-104),
// ensureRoute53 (route53.go:56-130) and CleanupRecordSet (:132-165).

// The owner-value rows of one object key, ascending by value row (= zone-major), fetched ONCE per object.  The
// first OWNED_CACHE rows are kept in registers/local memory; objects owning more fall back to re-walking the bucket.
constexpr u32 OWNED_CACHE = 8;
struct OwnedHit {
  u32 v, rec, zone;
  gar_str name;  // record name of the set that carries the value
};
struct Owned {
  OwnedHit hit[OWNED_CACHE];
  u32 n;  // total number of owned value rows (may exceed OWNED_CACHE)
  u64 okh;
  u32 kind;
  Str key;
};
GAR_HD bool owned_match(const DevTables &T, const IdxEntry &e, u32 kind, Str key) {
  return (e.a1 >> 31) == kind && streq(mkstr(T.a.slab, e.s0), key);
}
GAR_HD void owned_collect(const DevTables &T, const Work &W, u64 okh, u32 kind, Str key, Owned &o) {
  o.n = 0;
  o.okh = okh;
  o.kind = kind;
  o.key = key;
  Cursor c = idx_open(W.ix_val, okh);
  IdxEntry e;
  while (idx_next(W.ix_val, c, &e)) {
    if (!owned_match(T, e, kind, key)) continue;
    if (o.n < OWNED_CACHE) o.hit[o.n] = OwnedHit{e.row, e.a0, e.a1 & 0x3FFFFFFFu, e.s1};
    o.n++;
  }
}
GAR_HD void u_owned_collect(const DevTables &T, const Work &W, bool active, u64 okh, u32 kind, Str key, Owned &o) {
  if (active) {
    o.n = 0;
    o.okh = okh;
    o.kind = kind;
    o.key = key;
  }
  Cursor c = active ? idx_open(W.ix_val, okh) : Cursor{0, 0, 0};
  for (; GAR_ANY(c.pos < c.end);) {
    IdxEntry e;
    bool hit = false;
    if (c.pos < c.end) {
      e = load_entry(W.ix_val.ent + c.pos++);
      hit = e.tag == c.tag && (e.a1 >> 31) == kind;
    }
    if (u_streq(hit, hit ? mkstr(T.a.slab, e.s0) : Str{T.a.slab, 0}, key)) {
      if (o.n < OWNED_CACHE) o.hit[o.n] = OwnedHit{e.row, e.a0, e.a1 & 0x3FFFFFFFu, e.s1};
      o.n++;
    }
  }
}
GAR_HD OwnedHit owned_get(const DevTables &T, const Work &W, const Owned &o, u32 k) {
  if (k < OWNED_CACHE) return o.hit[k];
  Cursor c = idx_open(W.ix_val, o.okh);  // rare: re-walk the bucket to the k-th match
  IdxEntry e;
  u32 seen = 0;
  OwnedHit h{GAR_NONE, GAR_NONE, GAR_NONE, 0};
  while (idx_next(W.ix_val, c, &e)) {
    if (!owned_match(T, e, o.kind, o.key)) continue;
    if (seen++ == k) {
      h = OwnedHit{e.row, e.a0, e.a1 & 0x3FFFFFFFu, e.s1};
      break;
    }
  }
  return h;
}

// first alias record with type A under (zone, name): row and its alias DNSName ref  (rows of a bucket are ascending)
GAR_HD u32 first_alias_a(const DevTables &T, const Work &W, u32 zone, Str name, u64 name_hash, gar_str *alias_dns) {
  Cursor c = idx_open(W.ix_alias, key_hash_zoned_h(zone, name_hash));
  IdxEntry e;
  while (idx_next(W.ix_alias, c, &e)) {
    if (e.a0 != zone || e.a1 != GAR_RR_A) continue;
    if (streq(mkstr(T.a.slab, e.s0), name)) {
      *alias_dns = e.s1;
      return e.row;
    }
  }
  return GAR_NONE;
}
// smallest alias record row > after under (zone, name), any type
GAR_HD u32 next_alias_any(const DevTables &T, const Work &W, u32 zone, Str name, u32 after /* GAR_NONE = none yet */) {
  Cursor c = idx_open(W.ix_alias, key_hash_zoned(zone, name));
  IdxEntry e;
  while (idx_next(W.ix_alias, c, &e)) {
    if (after != GAR_NONE && e.row <= after) continue;
    if (e.a0 != zone) continue;
    if (streq(mkstr(T.a.slab, e.s0), name)) return e.row;
  }
  return GAR_NONE;
}

// CleanupRecordSet for one owner key: per zone, owned alias sets in record order, then owner metadata sets
GAR_HD void r53_cleanup(const DevTables &T, const Work &W, u32 obj, u32 kind, const Owned &ow, OpSink &s) {
  const gar_actual &A = T.a;
  u32 head = GAR_OP_HEAD(GAR_OP_R53_DELETE_RECORD, GAR_CTRL_R53, obj == GAR_NONE ? 0 : kind);
  u32 k = 0;
  while (k < ow.n) {  // value rows are ascending, i.e. grouped by zone in zone order
    u32 zone = owned_get(T, W, ow, k).zone;
    u32 kend = k;
    while (kend < ow.n && owned_get(T, W, ow, kend).zone == zone) kend++;
    // phase 0: repeatedly take the smallest not-yet-emitted alias record whose name is one of the zone group's names
    u32 last = GAR_NONE;
    for (;;) {
      u32 best = GAR_NONE, best_v = GAR_NONE;
      for (u32 x = k; x < kend; x++) {
        OwnedHit h = owned_get(T, W, ow, x);
        u32 r = next_alias_any(T, W, zone, mkstr(A.slab, h.name), last);
        // x ascending: the first value row that reaches a record is the one hostnameContains would hit first
        if (r != GAR_NONE && (best == GAR_NONE || r < best)) {
          best = r;
          best_v = h.v;
        }
      }
      if (best == GAR_NONE) break;
      s.put(head, obj, 0, zone, best, best_v);
      last = best;
    }
    // phase 1: one op per matching value of this zone
    for (u32 x = k; x < kend; x++) {
      OwnedHit h = owned_get(T, W, ow, x);
      s.put(head, obj, 1, zone, h.rec, h.v);
    }
    k = kend;
  }
}

// does the piece `hn` of strings.Split(all, ",") (a slice of `all`) also occur, byte for byte, earlier in the list?  (scalar)
GAR_HD bool piece_seen_before(Str all, Str hn) {
  u32 pos = 0;
  Str piece;
  while (next_piece(all, &pos, &piece)) {
    if (piece.p >= hn.p) return false;
    if (streq(piece, hn)) return true;
  }
  return false;
}

// Warp-synchronous like ga_reconcile: uniform loops over lbIngress index, hostname index and owned value rows; every
// probe and compare is a voted step.
GAR_HD u32 r53_reconcile(const DevTables &T, const Work &W, u32 i, bool valid, OpSink &s) {
  const gar_objects &o = T.o;
  const gar_actual &A = T.a;
  u32 result = GAR_STATUS(GAR_ST_IGNORED, 0, 0);
  u32 kind = 0, jb = 0, nj = 0;
  Str okey{T.o.slab, 0}, hostnames{T.o.slab, 0};
  u64 okh = 0;
  bool ensure = false;
  Owned ow;
  ow.n = 0;
  if (valid) {
    u32 dv = W.derived[i];
    if (dv & GAR_DV_R53_ELIGIBLE) {
      kind = o.obj_kind[i];
      okey = object_key(T, i);
      okh = W.okey_hash[i];
      if (!(dv & GAR_DV_R53_ANNOTATED)) {  // cleanup path: divergent, no votes inside
        owned_collect(T, W, okh, kind, okey, ow);
        r53_cleanup(T, W, i, kind, ow, s);
        result = GAR_STATUS(GAR_ST_OK, 0, GAR_EV_DELETED);
      } else {
        ensure = true;
        hostnames = mkstr(o.slab, W.ann_r53[i]);
        jb = o.obj_lbi_begin[i];
        nj = o.obj_lbi_begin[i + 1] - jb;
      }
    }
  }
  u32 ev = 0;
  bool stop = false, collected = false;
  // self-observation (include/garecon.h): a hostname this object visited before — earlier in the annotation or at an earlier
  // lbIngress — has its alias record in place, pointing at the accelerator of that visit
  bool have_prev = false;
  Str prev_acc_dns{A.slab, 0};
  for (u32 j = 0;; j++) {
    bool act = ensure && !stop && j < nj;
    if (!GAR_ANY(act)) break;
    bool probe = false;
    Str lbhost{o.slab, 0};
    if (act) {
      u32 code = W.tok_code[jb + j];
      if (code == GAR_TOK_PANIC) {
        result = GAR_STATUS(GAR_ST_PANIC, 0, ev);
        stop = true;
      } else if (code == GAR_TOK_NOT_AWS) {
      } else if (code >= GAR_TOK_ERR_NOT_ELB) {
        result = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_NOT_ELB + (code - GAR_TOK_ERR_NOT_ELB), ev);
        stop = true;
      } else {
        probe = true;
        lbhost = mkstr(o.slab, o.lbi_hostname[jb + j]);
      }
    }
    // ensureRoute53 (route53.go:56-130)
    u32 acc = GAR_NONE;
    gar_str acc_dns_ref = 0;
    u32 nacc = u_find_by_hostname(T, W, probe, lbhost, &acc, &acc_dns_ref);
    bool go = false;
    if (probe) {
      if (nacc > 1) {
        result = GAR_STATUS(GAR_ST_REQUEUE_60S, GAR_D_ACCEL_MANY, ev);
        stop = true;
      } else if (nacc == 0) {
        result = GAR_STATUS(GAR_ST_REQUEUE_60S, GAR_D_ACCEL_NONE, ev);
        stop = true;
      } else {
        go = true;
      }
    }
    Str acc_dns = go ? mkstr(A.slab, acc_dns_ref) : Str{A.slab, 0};
    if (GAR_ANY(go && !collected)) {  // the object's owner-value rows, fetched once (all lanes walk their bucket together)
      u_owned_collect(T, W, go && !collected, okh, kind, okey, ow);
      if (go) collected = true;
    }
    bool created = false;
    u32 pos = 0, k = 0;
    for (;;) {  // hostnames of the annotation, in order: strings.Split(annotation, ",")
      bool more = go && !stop && pos <= hostnames.n;
      if (!GAR_ANY(more)) break;
      u32 comma = u_find_byte(more, hostnames, pos, ',');
      Str hn = more ? substr(hostnames, pos, comma - pos) : Str{o.slab, 0};
      pos = comma + 1;
      u32 zone = u_find_hosted_zone(T, W, more, hn);
      if (more && zone == GAR_NONE) {
        result = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_NO_HOSTED_ZONE, ev);
        stop = true;
        more = false;
      }
      // findARecord over FindOwneredARecordSets: first (by record row) alias A record of the zone whose name is
      // owned by this object and unescapes to hostname + "."
      u32 rec = GAR_NONE;
      gar_str rec_alias = 0;
      for (u32 x = 0;; x++) {
        bool has = more && x < ow.n;
        if (!GAR_ANY(has)) break;
        Str nm{A.slab, 0};
        bool inzone = false;
        if (has) {
          OwnedHit h = owned_get(T, W, ow, x);
          inzone = h.zone == zone;
          if (inzone) nm = mkstr(A.slab, h.name);
        }
        bool cand = u_record_name_matches(inzone, nm, hn);
        gar_str al = 0;
        u32 r = u_first_alias_a(T, W, cand, zone, nm, &al);
        if (cand && r != GAR_NONE && (rec == GAR_NONE || r < rec)) {
          rec = r;
          rec_alias = al;
        }
      }
      // needRecordsUpdate (route53.go:373-381): *AliasTarget.DNSName != *accelerator.DnsName + "."
      bool have = more && rec != GAR_NONE;
      Str al = have ? mkstr(A.slab, rec_alias) : Str{A.slab, 0};
      bool shape = have && al.n == acc_dns.n + 1 && al.p[al.n - 1] == '.';
      bool same = u_streq(shape, substr(al, 0, shape ? acc_dns.n : 0), acc_dns);
      if (more) {
        if (!piece_seen_before(hostnames, hn)) {  // a repeated hostname was visited a moment ago with the same accelerator: in sync now
          if (!have_prev) {
            if (rec == GAR_NONE) {
              s.put(GAR_OP_HEAD(GAR_OP_R53_CREATE, GAR_CTRL_R53, kind), i, GAR_R53_SUB(j, k), zone, acc, GAR_NONE);
              created = true;
            } else if (!same) {
              s.put(GAR_OP_HEAD(GAR_OP_R53_UPSERT_A, GAR_CTRL_R53, kind), i, GAR_R53_SUB(j, k), zone, acc, rec);
            }
          } else if (!streq(acc_dns, prev_acc_dns)) {  // needRecordsUpdate only fires when the accelerator changed since the last visit
            s.put(GAR_OP_HEAD(GAR_OP_R53_UPSERT_A, GAR_CTRL_R53, kind), i, GAR_R53_SUB(j, k), zone, acc, rec == GAR_NONE ? GAR_PENDING : rec);
          }
        }
        k++;
      }
    }
    if (go && !stop && created) ev |= GAR_EV_CREATED;
    if (go && !stop) {
      have_prev = true;
      prev_acc_dns = acc_dns;
    }
  }
  if (ensure && !stop) result = GAR_STATUS(GAR_ST_OK, 0, ev);
  return result;
}

// ------------------------------------------------------------------ (a9) Route53 ensure, relational form
//
// The same decisions as r53_reconcile for the common shape (one lbIngress), split into uniform data-parallel steps:
//   link_value_alias  per owner value row : first alias A record under the same (zone, name)       [build side, once]
//   r53_prepare       per object          : filter, accelerator by target hostname, number of hostnames
//   r53_fill_pairs    per object          : (object, k, hostname slice) rows
//   r53_pair          per (object, k)     : GetHostedZone + findARecord over the object's owned names + needRecordsUpdate
//   r53_combine       per object          : replay the pair results in order (first NO_ZONE ends the stream), emit ops
// Objects of any other shape go through r53_reconcile inside r53_combine.

GAR_HD void link_value_alias(const DevTables &T, const Work &W, u32 v) {
  u32 row = GAR_NONE;
  gar_str dns = 0;
  if (W.val_cls[v] != VAL_NOT_OWNER) {
    u32 rec = W.val_rec[v];
    row = first_alias_a(T, W, W.rec_zone[rec], mkstr(T.a.slab, T.a.rec_name[rec]), W.rec_name_hash[rec], &dns);
  }
  ValLink l;
  l.alias_row = row;
  l.pad = 0;
  l.alias_dns = dns;
  W.val_link[v] = l;
}

// warp-synchronous.  Writes r53_mode, r53_acc, r53_acc_dns, pair count (into pair_begin[i]) and, for objects that
// are finished here, the status word.
GAR_HD void r53_prepare(const DevTables &T, const Work &W, u32 i, u32 t, bool valid, u32 *status) {
  const gar_objects &o = T.o;
  u32 mode = R53_MODE_DONE, st = GAR_STATUS(GAR_ST_IGNORED, 0, 0), npairs = 0;
  bool probe = false;
  Str lbhost{o.slab, 0}, hostnames{o.slab, 0};
  if (valid) {
    u32 dv = W.derived[i];
    if (dv & GAR_DV_R53_ELIGIBLE) {
      u32 jb = o.obj_lbi_begin[i], nj = o.obj_lbi_begin[i + 1] - jb;
      if (!(dv & GAR_DV_R53_ANNOTATED) || nj > 1) {
        mode = R53_MODE_OBJECT;
      } else if (nj == 0) {
        st = GAR_STATUS(GAR_ST_OK, 0, 0);  // annotated, no lbIngress: the loop body never runs (route53/service.go:73)
      } else {
        u32 code = W.tok_code[jb];
        if (code == GAR_TOK_PANIC) st = GAR_STATUS(GAR_ST_PANIC, 0, 0);
        else if (code == GAR_TOK_NOT_AWS) st = GAR_STATUS(GAR_ST_OK, 0, 0);
        else if (code >= GAR_TOK_ERR_NOT_ELB) st = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_NOT_ELB + (code - GAR_TOK_ERR_NOT_ELB), 0);
        else {
          probe = true;
          lbhost = mkstr(o.slab, o.lbi_hostname[jb]);
          hostnames = mkstr(o.slab, W.ann_r53[i]);
        }
      }
    }
  }
  u32 acc = GAR_NONE;
  gar_str acc_dns = 0;
  u32 nacc = u_find_by_hostname(T, W, probe, lbhost, &acc, &acc_dns);
  bool go = false;
  if (probe) {
    if (nacc > 1) st = GAR_STATUS(GAR_ST_REQUEUE_60S, GAR_D_ACCEL_MANY, 0);
    else if (nacc == 0) st = GAR_STATUS(GAR_ST_REQUEUE_60S, GAR_D_ACCEL_NONE, 0);
    else go = true;
  }
  // number of pieces of strings.Split(annotation, ",") = commas + 1
  u32 pos = 0;
  for (;;) {
    bool more = go && pos <= hostnames.n;
    if (!GAR_ANY(more)) break;
    u32 comma = u_find_byte(more, hostnames, pos, ',');
    if (more) {
      npairs++;
      pos = comma + 1;
    }
  }
  if (go) mode = R53_MODE_PAIRS;
  if (valid) {
    W.r53_mode[i] = (u8)mode;
    W.r53_acc[i] = acc;
    W.r53_acc_dns[i] = acc_dns;
    W.pair_begin[t] = npairs;
    if (mode == R53_MODE_DONE) status[t] = st;
  }
}

GAR_HD void r53_fill_pairs(const DevTables &T, const Work &W, u32 i, u32 t) {
  if (W.r53_mode[i] != R53_MODE_PAIRS) return;
  gar_str ref = W.ann_r53[i];
  Str hostnames = mkstr(T.o.slab, ref);
  u32 p = W.pair_begin[t], pos = 0, np = 0;
  u32 st[8], ln[8];  // the first pieces, for the repeat check (annotations with more hostnames fall back to a re-scan)
  Str piece;
  while (next_piece(hostnames, &pos, &piece)) {
    if (p >= W.pair_cap) break;  // more pairs than the arrays hold: the diff is re-run with larger ones
    W.pair_obj[p] = i;
    W.pair_hn[p] = GAR_STR(GAR_STR_OFF(ref) + (u64)(piece.p - hostnames.p), piece.n);
    // self-observation (include/garecon.h): a repeated hostname needs no evaluation — the annotation bytes are in hand here
    bool repeat = false;
    for (u32 q = 0; q < np && q < 8 && !repeat; q++) repeat = ln[q] == piece.n && streq(substr(hostnames, st[q], ln[q]), piece);
    if (!repeat && np > 8) repeat = piece_seen_before(hostnames, piece);
    W.pair_code[p] = repeat ? (u8)PAIR_REPEAT : (u8)PAIR_IN_SYNC;
    if (np < 8) {
      st[np] = (u32)(piece.p - hostnames.p);
      ln[np] = piece.n;
    }
    np++;
    p++;
  }
}

// warp-synchronous; one lane per (object, hostname)
GAR_HD void r53_pair(const DevTables &T, const Work &W, u32 p, bool valid) {
  const gar_actual &A = T.a;
  u32 i = 0, kind = 0;
  Str hn{T.o.slab, 0}, okey{T.o.slab, 0};
  u64 okh = 0;
  valid = valid && W.pair_code[p] != PAIR_REPEAT;
  if (valid) {
    i = W.pair_obj[p];
    hn = mkstr(T.o.slab, W.pair_hn[p]);
    kind = T.o.obj_kind[i];
    okey = object_key(T, i);
    okh = W.okey_hash[i];
  }
  u32 zone = u_find_hosted_zone(T, W, valid, hn);
  bool live = valid && zone != GAR_NONE;
  // findARecord over FindOwneredARecordSets: among the owner-value rows of this object in `zone` whose record name
  // unescapes to hostname + ".", the smallest first-alias-A row (route53.go:216-238,360-367)
  u32 rec = GAR_NONE;
  gar_str rec_alias = 0;
  Cursor c = u_open(W.ix_val, live, okh);
  for (; GAR_ANY(c.pos < c.end);) {
    IdxEntry e;
    bool hit = false;
    if (c.pos < c.end) {
      e = load_entry(W.ix_val.ent + c.pos++);
      hit = e.tag == c.tag && (e.a1 >> 31) == kind && (e.a1 & 0x3FFFFFFFu) == zone;
    }
    bool mine = u_streq(hit, hit ? mkstr(A.slab, e.s0) : Str{A.slab, 0}, okey);
    Str nm = mine ? mkstr(A.slab, e.s1) : Str{A.slab, 0};
    bool plain = mine && !(e.a1 & VALNAME_HAS_BACKSLASH);
    bool shape = plain && nm.n == hn.n + 1 && nm.p[nm.n - 1] == '.';
    bool match = u_streq(shape, substr(nm, 0, shape ? hn.n : 0), hn);
    if (mine && !plain) match = record_name_matches(nm, hn);  // possible \052 escape: scalar, rare
    if (match) {
      ValLink l = W.val_link[e.row];
      if (l.alias_row != GAR_NONE && (rec == GAR_NONE || l.alias_row < rec)) {
        rec = l.alias_row;
        rec_alias = l.alias_dns;
      }
    }
  }
  // needRecordsUpdate (route53.go:373-381)
  bool have = live && rec != GAR_NONE;
  Str acc_dns = have ? mkstr(A.slab, W.r53_acc_dns[i]) : Str{A.slab, 0};
  Str al = have ? mkstr(A.slab, rec_alias) : Str{A.slab, 0};
  bool shape = have && al.n == acc_dns.n + 1 && al.p[al.n - 1] == '.';
  bool same = u_streq(shape, substr(al, 0, shape ? acc_dns.n : 0), acc_dns);
  if (valid) {
    u32 code = !live ? PAIR_NO_ZONE : rec == GAR_NONE ? PAIR_CREATE : same ? PAIR_IN_SYNC : PAIR_UPSERT;
    W.pair_code[p] = (u8)code;
    W.pair_zone[p] = zone;
    W.pair_rec[p] = rec;
  }
}

// warp-synchronous (objects in R53_MODE_OBJECT call the voted r53_reconcile)
GAR_HD u32 r53_combine(const DevTables &T, const Work &W, u32 i, u32 t, bool valid, u32 prev_status, OpSink &s) {
  u32 mode = valid ? W.r53_mode[i] : R53_MODE_DONE;
  u32 st = prev_status;
  bool slow = mode == R53_MODE_OBJECT;
  if (GAR_ANY(slow)) {
    u32 r = r53_reconcile(T, W, i, slow, s);
    if (slow) st = r;
  }
  if (mode == R53_MODE_PAIRS) {
    u32 kind = T.o.obj_kind[i], acc = W.r53_acc[i];
    bool created = false, stop = false;
    u32 k = 0;
    for (u32 p = W.pair_begin[t]; p < W.pair_begin[t + 1] && p < W.pair_cap && !stop; p++, k++) {
      u32 code = W.pair_code[p];
      if (code == PAIR_NO_ZONE) {
        st = GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_NO_HOSTED_ZONE, 0);
        stop = true;
      } else if (code == PAIR_CREATE) {
        s.put(GAR_OP_HEAD(GAR_OP_R53_CREATE, GAR_CTRL_R53, kind), i, GAR_R53_SUB(0, k), W.pair_zone[p], acc, GAR_NONE);
        created = true;
      } else if (code == PAIR_UPSERT) {
        s.put(GAR_OP_HEAD(GAR_OP_R53_UPSERT_A, GAR_CTRL_R53, kind), i, GAR_R53_SUB(0, k), W.pair_zone[p], acc, W.pair_rec[p]);
      }
    }
    if (!stop) st = GAR_STATUS(GAR_ST_OK, 0, created ? GAR_EV_CREATED : 0);
  }
  return st;
}

// ------------------------------------------------------------------ orphans (delete events of keys that left the cache)

GAR_HD bool object_in_cache(const DevTables &T, const Work &W, u32 kind, Str key, u64 key_hash) {
  Cursor c = idx_open(W.ix_obj, key_hash);
  IdxEntry e;
  while (idx_next(W.ix_obj, c, &e))
    if (e.a0 == kind && streq(mkstr(T.o.slab, e.s0), key)) return true;
  return false;
}

// process{Service,Ingress}Delete of the globalaccelerator controller (service.go:28-52, ingress.go:29-54) for an
// accelerator whose owner key has no object: returns 1 and emits the delete op
GAR_HD u32 ga_orphan(const DevTables &T, const Work &W, u32 acc, OpSink &s) {
  if (acc >= W.acc_guest_from) return 0;
  if (W.acc_claimed && W.acc_claimed[acc]) return 0;  // its owner's object iterated it: the object is in the cache
  u32 fl = W.acc_flags[acc];
  if (!(fl & ACC_MINE) || !(fl & ACC_OWNER_3PART)) return 0;
  u32 kind = (fl & ACC_OWNER_INGRESS) ? 1u : 0u;
  if (object_in_cache(T, W, kind, mkstr(T.a.slab, W.acc_owner_key[acc]), W.acc_owner_hash[acc])) return 0;
  put_delete_chain(T, s, GAR_NONE, 0, acc);
  return 1;
}

// is value row v an owner value of this cluster whose object left the cache?
GAR_HD void mark_orphan_value(const DevTables &T, const Work &W, u32 v) {
  u32 cls = W.val_cls[v];
  u8 orphan = 0;
  if (cls & VAL_OWNER_3PART) {
    u32 kind = (cls & VAL_OWNER_INGRESS) ? 1u : 0u;
    orphan = object_in_cache(T, W, kind, mkstr(T.a.slab, W.val_key[v]), W.val_key_hash[v]) ? 0 : 1;
  }
  if (orphan) {
    u32 rec = W.val_rec[v];
    ix_count(W.hist[IX_OVN], key_hash_zoned_h(W.rec_zone[rec], W.rec_name_hash[rec]));
  }
  W.val_orphan[v] = orphan;
}

// phase 0 of the orphan section for alias record r: one op per distinct orphan owner value that has a value
// row under the same (zone, name); a2 = the first such value row.  Rows of ix_ovn buckets are ascending.
GAR_HD void r53_orphan_alias(const DevTables &T, const Work &W, u32 r, OpSink &s) {
  const gar_actual &A = T.a;
  if (!A.rec_has_alias[r]) return;
  u32 zone = W.rec_zone[r];
  Str name = mkstr(A.slab, A.rec_name[r]);
  u64 h = key_hash_zoned_h(zone, W.rec_name_hash[r]);
  Cursor c = idx_open(W.ix_ovn, h);
  IdxEntry e;
  while (idx_next(W.ix_ovn, c, &e)) {
    if (e.a1 != zone || !streq(mkstr(A.slab, e.s0), name)) continue;
    // skip if an earlier row of the bucket carries the same value under the same name
    Str val = mkstr(A.slab, e.s1);
    bool dup = false;
    Cursor c2 = idx_open(W.ix_ovn, h);
    IdxEntry e2;
    while (idx_next(W.ix_ovn, c2, &e2) && e2.row < e.row) {
      if (e2.a1 == zone && streq(mkstr(A.slab, e2.s0), name) && streq(mkstr(A.slab, e2.s1), val)) {
        dup = true;
        break;
      }
    }
    if (dup) continue;
    s.put(GAR_OP_HEAD(GAR_OP_R53_DELETE_RECORD, GAR_CTRL_R53, 0), GAR_NONE, 0, zone, r, e.row);
  }
}

// ------------------------------------------------------------------ (f3) EndpointGroupBinding set-diff
//
// pkg/controller/endpointgroupbinding/reconcile.go:20-217.  One thread per binding (bindings are few); uses the
// snapshot's object index, tokeniser output and LB index.

struct DevBindings {
  gar_bindings b;     // device pointers
  HashIdx ix_eg;      // endpoint-group ARN -> known_eg row
};

GAR_HD bool egb_eg_exists(const DevBindings &B, Str arn) {
  Cursor c = idx_open(B.ix_eg, gar_hash(arn));
  IdxEntry e;
  while (idx_next(B.ix_eg, c, &e))
    if (streq(mkstr(B.b.slab, e.s0), arn)) return true;
  return false;
}

// the LB row a lbIngress row resolves to: GetLBNameFromHostname + GetLoadBalancer (reconcile.go:125-138); *detail != 0 on error
GAR_HD u32 egb_lb_of(const DevTables &T, const Work &W, u32 lbi_row, u32 *detail) {
  u32 code = W.tok_code[lbi_row];
  *detail = 0;
  if (code == GAR_TOK_NOT_AWS || code == GAR_TOK_PANIC) {  // no DetectCloudProvider on this path: both regexps simply do not match
    *detail = GAR_D_NOT_ELB;
    return GAR_NONE;
  }
  if (code >= GAR_TOK_ERR_NOT_ELB) {
    *detail = GAR_D_NOT_ELB + (code - GAR_TOK_ERR_NOT_ELB);
    return GAR_NONE;
  }
  u32 st;
  u32 lb = find_lb(T, W, mkstr(T.o.slab, W.tok_region[lbi_row]), mkstr(T.o.slab, W.tok_name[lbi_row]), &st);
  if (lb == GAR_NONE) *detail = GAR_D_LB_NOT_FOUND;
  return lb;
}

GAR_HD u32 egb_reconcile(const DevTables &T, const Work &W, const DevBindings &B, u32 k, OpSink &s) {
  const gar_bindings &b = B.b;
  const gar_actual &A = T.a;
  u32 flags = b.egb_flags[k];
  u32 eb = b.egb_ep_begin[k], n = b.egb_ep_begin[k + 1] - eb;
  Str eg_arn = mkstr(b.slab, b.egb_eg_arn[k]);
  auto H = [](u32 op) { return GAR_OP_HEAD(op, GAR_CTRL_EGB, 0); };
  if (flags & GAR_EGB_DELETING) {  // reconcileDelete (:35-96)
    if (n == 0 || !egb_eg_exists(B, eg_arn)) {
      s.put(H(GAR_OP_EGB_REMOVE_FINALIZER), k, 0, GAR_NONE, GAR_NONE, GAR_NONE);
      return GAR_STATUS(GAR_ST_OK, 0, 0);
    }
    // `endpointIds` aliases obj.Status.EndpointIds while the loop indexes the latter (:70-85): iteration i sees the element
    // that started at index min(2i, n-1), and `endpointIds[i+1:]` panics as soon as i+1 exceeds the shrinking length
    u32 len = n;
    for (u32 i = 0; i < n; i++) {
      u32 src = 2 * i < n - 1 ? 2 * i : n - 1;
      s.put(H(GAR_OP_EGB_REMOVE_ENDPOINT), k, 0, eb + src, GAR_NONE, GAR_NONE);
      if (i + 1 > len) return GAR_STATUS(GAR_ST_PANIC, 0, 0);
      len--;
    }
    s.put(H(GAR_OP_EGB_UPDATE_STATUS), k, 0, GAR_NONE, GAR_NONE, GAR_NONE);
    return GAR_STATUS(GAR_ST_REQUEUE_1S, 0, 0);
  }
  if (!(flags & GAR_EGB_HAS_FINALIZERS)) {  // reconcileCreate (:98-110)
    s.put(H(GAR_OP_EGB_ADD_FINALIZER), k, 0, GAR_NONE, GAR_NONE, GAR_NONE);
    return GAR_STATUS(GAR_ST_OK, 0, 0);
  }
  // reconcileUpdate (:112-217).  getLoadBalancerHostName (:219-252)
  u32 jb = 0, nj = 0;
  u32 refkind = b.egb_ref_kind[k];
  if (refkind != GAR_EGB_REF_NONE) {
    u32 kind = refkind == GAR_EGB_REF_SERVICE ? GAR_KIND_SERVICE : GAR_KIND_INGRESS;
    Str key = mkstr(b.slab, b.egb_ref_key[k]);
    Cursor c = idx_open(W.ix_obj, key_hash_kinded(kind, key));
    IdxEntry e;
    u32 obj = GAR_NONE;
    while (idx_next(W.ix_obj, c, &e))
      if (e.a0 == kind && streq(mkstr(T.o.slab, e.s0), key)) {
        obj = e.row;
        break;
      }
    if (obj == GAR_NONE) return GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_REF_NOT_FOUND, 0);
    jb = T.o.obj_lbi_begin[obj];
    nj = T.o.obj_lbi_begin[obj + 1] - jb;
  }
  for (u32 j = 0; j < nj; j++) {  // every hostname must resolve before anything is decided (:124-139)
    u32 detail;
    if (egb_lb_of(T, W, jb + j, &detail) == GAR_NONE) return GAR_STATUS(GAR_ST_ERR_RETRY, detail, 0);
  }
  // the `arns` map: ARN -> LB name.  first(j): hostname j is the first one with its ARN.
  auto arn_of = [&](u32 j) {
    u32 d;
    return mkstr(A.slab, A.lb_arn[egb_lb_of(T, W, jb + j, &d)]);
  };
  auto is_first = [&](u32 j) {
    Str a = arn_of(j);
    for (u32 i = 0; i < j; i++)
      if (streq(arn_of(i), a)) return false;
    return true;
  };
  auto in_status = [&](Str a) {
    for (u32 x = 0; x < n; x++)
      if (streq(mkstr(b.slab, b.ep_id[eb + x]), a)) return true;
    return false;
  };
  auto in_arns = [&](Str id) {
    for (u32 j = 0; j < nj; j++)
      if (streq(arn_of(j), id)) return true;
    return false;
  };
  u32 nnew = 0, nrem = 0;
  for (u32 j = 0; j < nj; j++)
    if (is_first(j) && !in_status(arn_of(j))) nnew++;
  for (u32 x = 0; x < n; x++)
    if (!in_arns(mkstr(b.slab, b.ep_id[eb + x]))) nrem++;
  if (nnew == 0 && nrem == 0 && (flags & GAR_EGB_OBSERVED)) return GAR_STATUS(GAR_ST_OK, 0, 0);
  if (!egb_eg_exists(B, eg_arn)) return GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_EG_NOT_FOUND, 0);
  if (nrem > 0 && nj == 0) return GAR_STATUS(GAR_ST_PANIC, 0, 0);  // regionalCloud is nil (:121,:160)
  for (u32 x = 0; x < n; x++)
    if (!in_arns(mkstr(b.slab, b.ep_id[eb + x]))) s.put(H(GAR_OP_EGB_REMOVE_ENDPOINT), k, 0, eb + x, GAR_NONE, GAR_NONE);
  // AddLBToEndpointGroup looks the LB up again by NAME in the region of the LAST hostname (:122-131,:172; global_accelerator.go:572-591)
  Str last_region = nj ? mkstr(T.o.slab, W.tok_region[jb + nj - 1]) : Str{T.o.slab, 0};
  for (u32 j = 0; j < nj; j++) {
    if (!is_first(j) || in_status(arn_of(j))) continue;
    u32 jl = j;  // arns[arn] holds the name written by the LAST hostname with this ARN
    for (u32 i = j + 1; i < nj; i++)
      if (streq(arn_of(i), arn_of(j))) jl = i;
    u32 st;
    u32 lb2 = find_lb(T, W, last_region, mkstr(T.o.slab, W.tok_name[jb + jl]), &st);
    if (lb2 == GAR_NONE) return GAR_STATUS(GAR_ST_ERR_RETRY, GAR_D_LB_NOT_FOUND, 0);
    if (st != GAR_LB_ACTIVE) return GAR_STATUS(GAR_ST_REQUEUE_30S, 0, 0);
    s.put(H(GAR_OP_EGB_ADD_ENDPOINT), k, 0, lb2, GAR_NONE, GAR_NONE);
  }
  for (u32 j = 0; j < nj; j++)
    if (is_first(j)) {
      u32 d;
      s.put(H(GAR_OP_EGB_UPDATE_WEIGHT), k, 0, egb_lb_of(T, W, jb + j, &d), GAR_NONE, GAR_NONE);
    }
  s.put(H(GAR_OP_EGB_UPDATE_STATUS), k, 0, GAR_NONE, GAR_NONE, GAR_NONE);
  return GAR_STATUS(GAR_ST_OK, 0, 0);
}
