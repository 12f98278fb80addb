/*
 * garecon.h — C ABI of the B200 batch reconcile-diff engine (libgarecon.so).
 *
 * Drop-in boundary for ONE path of h3poteto/aws-global-accelerator-controller: the
 * desired-vs-actual decision logic that the Go controller runs per work item behind
 *   pkg/reconcile/reconcile.go:22-26   (KeyToObjFunc / ProcessDeleteFunc / ProcessCreateOrUpdateFunc,
 *                                       ProcessNextWorkItem)
 * and that bottoms out in the decision functions of pkg/cloudprovider/aws
 * (global_accelerator.go:31-570, route53.go:18-130,216-238,335-395, load_balancer.go:32-93) and
 * pkg/cloudprovider/provider.go:8-17.
 *
 * The reference has no FFI (CGO_ENABLED="0", Makefile:27); these entry points are what a cgo shim
 * for that path would bind (see INTEGRATION.md).  Plain pointers and sizes only: no C++ / torch types.
 *
 * Data model
 * ----------
 * Everything is struct-of-arrays.  Strings never travel as pointers: a string is a `gar_str`
 * (40-bit byte offset | 24-bit length) into the byte slab of the table group it belongs to
 * (`gar_objects.slab` or `gar_actual.slab`).  One-to-many relations are CSR: `x_begin[i] .. x_begin[i+1]`
 * indexes the child table, every `*_begin` array has n+1 entries.  Child rows keep the order in which
 * the reference would see them (map-free lists in API/list order): that order is part of the contract
 * because the change set is ordered.
 *
 * Ownership: the caller owns every input buffer and may free it as soon as gar_snapshot_load returns
 * (cgo must not let C retain Go pointers); the engine owns a change set until gar_changeset_free.
 * Errors: every call returns GAR_OK or a negative gar_rc; gar_last_error gives the text.  The engine
 * never aborts and has no CPU fallback: without a usable sm_100 device every call fails.
 * Threading: calls on one engine are serialised by an internal mutex and may come from any OS thread.
 */
#ifndef GARECON_H
#define GARECON_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GAR_ABI_VERSION 1u

/* ---------------------------------------------------------------- strings */

typedef uint64_t gar_str; /* bits 0..39 byte offset into the slab, bits 40..63 length in bytes */
#define GAR_STR_OFF_BITS 40
#define GAR_STR(off, len) (((uint64_t)(len) << GAR_STR_OFF_BITS) | (uint64_t)(off))
#define GAR_STR_OFF(s) ((uint64_t)(s) & ((1ull << GAR_STR_OFF_BITS) - 1))
#define GAR_STR_LEN(s) ((uint32_t)((uint64_t)(s) >> GAR_STR_OFF_BITS))
#define GAR_NONE 0xFFFFFFFFu /* "no row" in op arguments */
#define GAR_PENDING 0xFFFFFFFEu /* op argument: the resource an EARLIER op of the same object creates (see "Self-observation") */

/* ---------------------------------------------------------------- return codes */

typedef enum {
  GAR_OK = 0,
  GAR_E_INVALID = -1,  /* bad argument / malformed table (offset out of slab, non-monotone CSR ...) */
  GAR_E_NO_DEVICE = -2,/* no CUDA device, or device is not sm_100 */
  GAR_E_CUDA = -3,     /* a CUDA call failed; text in gar_last_error */
  GAR_E_STATE = -4,    /* call order wrong (diff before load ...) */
  GAR_E_NOMEM = -5
} gar_rc;

/* ---------------------------------------------------------------- desired side: the informer cache */

/* obj_kind — which lister the row came from (globalaccelerator/controller.go:39,41) */
enum { GAR_KIND_SERVICE = 0, GAR_KIND_INGRESS = 1 };
/* obj_spec_type — corev1.ServiceType, Service rows only (globalaccelerator/service.go:19) */
enum { GAR_SVC_CLUSTERIP = 0, GAR_SVC_NODEPORT = 1, GAR_SVC_LOADBALANCER = 2, GAR_SVC_EXTERNALNAME = 3 };
/* obj_flags */
enum {
  GAR_OBJ_HAS_LB_CLASS = 1u << 0,      /* Service: spec.loadBalancerClass != nil (service.go:20) */
  GAR_OBJ_HAS_INGRESS_CLASS = 1u << 1  /* Ingress: spec.ingressClassName != nil; value in obj_ingress_class (ingress.go:20) */
};

typedef struct gar_objects {
  uint32_t n_objects;
  const uint8_t *obj_kind;          /* [n] GAR_KIND_* */
  const uint8_t *obj_spec_type;     /* [n] GAR_SVC_* (0 for Ingress rows) */
  const uint8_t *obj_flags;         /* [n] GAR_OBJ_* */
  const gar_str *obj_ns;            /* [n] metadata.namespace */
  const gar_str *obj_name;          /* [n] metadata.name */
  const gar_str *obj_ingress_class; /* [n] *spec.ingressClassName (only if GAR_OBJ_HAS_INGRESS_CLASS) */
  const uint32_t *obj_ann_begin;    /* [n+1] -> ann_*: metadata.annotations (keys unique per object) */
  const uint32_t *obj_lbi_begin;    /* [n+1] -> lbi_*: status.loadBalancer.ingress[] in order */
  const uint32_t *obj_port_begin;   /* [n+1] -> port_*: Service: spec.ports[] in order (global_accelerator.go:506);
                                       Ingress: defaultBackend.service.port.number (if defaultBackend and its
                                       .service are set) followed by every rules[].http.paths[].backend.service
                                       .port.number in order (global_accelerator.go:544-555; named ports are 0) */
  uint32_t n_ann;
  const gar_str *ann_key;           /* [n_ann] */
  const gar_str *ann_val;           /* [n_ann] */
  uint32_t n_lbi;
  const gar_str *lbi_hostname;      /* [n_lbi] status.loadBalancer.ingress[].hostname ("" when only .ip is set) */
  uint32_t n_ports;
  const int32_t *port_number;       /* [n_ports] */
  const gar_str *port_proto;        /* [n_ports] Service: spec.ports[].protocol as written ("TCP","UDP",...); Ingress: len 0 */
  const uint8_t *slab;
  uint64_t slab_len;
} gar_objects;

/* ---------------------------------------------------------------- actual side: listed AWS snapshots */

/* lb_state — elbv2types.LoadBalancerStateEnum (global_accelerator.go:125) */
enum { GAR_LB_ACTIVE = 0, GAR_LB_PROVISIONING = 1, GAR_LB_ACTIVE_IMPAIRED = 2, GAR_LB_FAILED = 3 };
/* lis_proto — gatypes.Protocol */
enum { GAR_PROTO_TCP = 0, GAR_PROTO_UDP = 1 };
/* rec_type — route53types.RRType; only A is distinguished by the path (route53.go:362) */
enum { GAR_RR_OTHER = 0, GAR_RR_A = 1, GAR_RR_TXT = 2, GAR_RR_CNAME = 3, GAR_RR_AAAA = 4 };

/* Only columns the decisions read are part of the ABI.  Identifiers the executor needs to CALL AWS with
   (accelerator / listener / endpoint-group ARNs, hosted-zone ids) stay on the Go side, addressed by the row
   indices the ops carry. */
typedef struct gar_actual {
  /* ELBv2 DescribeLoadBalancers, every region listed (load_balancer.go:13-30).  A lookup is by
     (region, name); with duplicates the first row wins, as `range res.LoadBalancers` does. */
  uint32_t n_lbs;
  const gar_str *lb_region;
  const gar_str *lb_name;
  const gar_str *lb_dns;
  const gar_str *lb_arn;
  const uint8_t *lb_state;
  /* Global Accelerator: ListAccelerators order (global_accelerator.go:624-641) */
  uint32_t n_accels;
  const gar_str *acc_name;
  const gar_str *acc_dns;
  const uint8_t *acc_enabled;
  const uint32_t *acc_tag_begin;   /* [n_accels+1] -> tag_*: ListTagsForResource order (:643-652) */
  const uint32_t *acc_lis_begin;   /* [n_accels+1] -> lis_*: ListListeners(accelerator) order (:789-803) */
  uint32_t n_tags;
  const gar_str *tag_key;
  const gar_str *tag_val;
  uint32_t n_listeners;
  const uint8_t *lis_proto;
  const uint32_t *lis_pr_begin;    /* [n_listeners+1] -> pr_from: Listener.PortRanges[] */
  const uint32_t *lis_eg_begin;    /* [n_listeners+1] -> eg_*: ListEndpointGroups(listener) order (:885-898) */
  uint32_t n_port_ranges;
  const int32_t *pr_from;          /* PortRange.FromPort — the only field the comparison reads (:460-462) */
  uint32_t n_egs;
  const uint32_t *eg_ep_begin;     /* [n_egs+1] -> ep_id: EndpointDescriptions[] */
  uint32_t n_endpoints;
  const gar_str *ep_id;            /* EndpointDescription.EndpointId (:496) */
  /* Route53: ListHostedZones order (route53.go:199-214); records in ListResourceRecordSets order (:317-333).
     A by-name zone lookup takes the first row whose name matches exactly (:349-353). */
  uint32_t n_zones;
  const gar_str *zone_name;        /* with trailing dot, as AWS returns it */
  const uint32_t *zone_rec_begin;  /* [n_zones+1] -> rec_* */
  uint32_t n_records;
  const gar_str *rec_name;         /* as AWS returns it: trailing dot, '*' escaped as \052 */
  const uint8_t *rec_type;         /* GAR_RR_* */
  const uint8_t *rec_has_alias;    /* AliasTarget != nil */
  const gar_str *rec_alias_dns;    /* AliasTarget.DNSName (only if rec_has_alias) */
  const uint32_t *rec_val_begin;   /* [n_records+1] -> val_value: ResourceRecords[] */
  uint32_t n_values;
  const gar_str *val_value;        /* ResourceRecord.Value (TXT values keep their double quotes) */
  const uint8_t *slab;
  uint64_t slab_len;
} gar_actual;

/* ---------------------------------------------------------------- engine configuration */

typedef struct gar_config {
  uint32_t abi_version;      /* GAR_ABI_VERSION */
  int32_t device;            /* CUDA device ordinal */
  const char *cluster_name;  /* --cluster-name (cmd/controller/controller.go:33); NUL-terminated, copied */
  uint32_t flags;            /* GAR_FLAG_* */
} gar_config;
#define GAR_FLAG_STAGE_TIMING 1u /* bracket every stage with CUDA events; read them with gar_last_stage_timings */
#define GAR_FLAG_REPREPARE 2u    /* rebuild the snapshot's digests and hash indexes on EVERY diff instead of once per load:
                                    for measuring the complete pipeline (bench.py "value", ncu captures) */
#define GAR_FLAG_NO_ORPHANS 4u   /* gar_diff leaves the two orphan sections empty: nothing is ever deleted on the strength of a key being
                                    ABSENT from the object table.  Deletes then come only from objects in the table (unmanaged / de-annotated)
                                    and from keys passed explicitly to gar_diff_keys as deleted (the reference's own rule: cleanup runs on an
                                    observed delete event, globalaccelerator/controller.go:113-173) */
#define GAR_FLAG_ALLOW_EMPTY_CACHE 8u /* see "Orphan sweep precondition" below */
/* Orphan sweep precondition.  The orphan sections of gar_diff stand for the delete events of every owner key that is tagged on an
   AWS resource of this cluster but has no object in the table: they are only right when the table is the COMPLETE, SYNCED informer
   cache of the whole cluster (HasSynced() true on both informers, no namespace-scoped cache, no failed or partial list, all slices
   present in sharded mode).  A caller that cannot guarantee that must set GAR_FLAG_NO_ORPHANS.  As a last line of defence gar_diff
   refuses (GAR_E_STATE) to emit orphan deletes when the object table is EMPTY while owned resources exist — the signature of an
   informer that has not synced — unless GAR_FLAG_ALLOW_EMPTY_CACHE says the empty cache is real (the last object was deleted). */

/* ---------------------------------------------------------------- output: the change set */

/* Per (controller, object) status word:  bits 0..7 gar_status, bits 8..15 gar_detail, bits 16..23 gar_event */
typedef enum {
  GAR_ST_IGNORED = 0,     /* object fails the controller's event filter (service.go:18-26, ingress.go:19-27) */
  GAR_ST_OK = 1,          /* Result{}, nil -> Forget (reconcile.go:87-89) */
  GAR_ST_SKIP_NO_LB = 2,  /* status.loadBalancer.ingress empty (service.go:59-62): Result{}, nil */
  GAR_ST_REQUEUE_30S = 3, /* LB not active (global_accelerator.go:125-128) -> AddAfter(30s) */
  GAR_ST_REQUEUE_60S = 4, /* accelerator-by-hostname count != 1 (route53.go:68-77) -> AddAfter(1m) */
  GAR_ST_ERR_RETRY = 5,   /* error, not NoRetry -> AddRateLimited (reconcile.go:75-77) */
  GAR_ST_ERR_NORETRY = 6, /* *NoRetryError -> dropped (reconcile.go:73-74); not produced by a snapshot diff */
  GAR_ST_PANIC = 7        /* DetectCloudProvider indexes parts[len-2] of a <2-label hostname (provider.go:9-10) */
} gar_status;

typedef enum {
  GAR_D_NONE = 0,
  GAR_D_NOT_ELB = 1,            /* load_balancer.go:42 */
  GAR_D_PARSE_INTERNAL_ALB = 2, /* load_balancer.go:64 */
  GAR_D_PARSE_PUBLIC_ALB = 3,   /* load_balancer.go:73 */
  GAR_D_PARSE_NLB = 4,          /* load_balancer.go:90 */
  GAR_D_LB_NOT_FOUND = 5,       /* load_balancer.go:29 (or the API's LoadBalancerNotFound) */
  GAR_D_LB_DNS_MISMATCH = 6,    /* global_accelerator.go:122-124 */
  GAR_D_TOO_MANY_LISTENERS = 7, /* global_accelerator.go:808-810 */
  GAR_D_TOO_MANY_EGS = 8,       /* global_accelerator.go:902-904 */
  GAR_D_NO_HOSTED_ZONE = 9,     /* route53.go:338-340 */
  GAR_D_ACCEL_MANY = 10,        /* route53.go:68-72 */
  GAR_D_ACCEL_NONE = 11         /* route53.go:73-77 */
} gar_detail;

enum {
  GAR_EV_CREATED = 1u << 0, /* GlobalAcceleratorCreated / Route53RecordCreated event (service.go:116-118, route53/service.go:101-103) */
  GAR_EV_DELETED = 1u << 1  /* GlobalAcceleratorDeleted / Route53RecordDeleted event (service.go:82, route53/service.go:67) */
};
#define GAR_STATUS(st, detail, ev) ((uint32_t)(st) | ((uint32_t)(detail) << 8) | ((uint32_t)(ev) << 16))
#define GAR_STATUS_CODE(w) ((w) & 0xFFu)
#define GAR_STATUS_DETAIL(w) (((w) >> 8) & 0xFFu)
#define GAR_STATUS_EVENT(w) (((w) >> 16) & 0xFFu)

/* Op codes.  Every op stands for a mutation the reference performs in-line.  Arguments are row indices
   into the input tables (GAR_NONE = absent).  `obj` is GAR_NONE for orphan ops.
     op                    sub            a0      a1               a2
     GA_CREATE_CHAIN       j              lb      NONE             NONE     global_accelerator.go:136-148,213-232
     GA_UPDATE_ACCEL       j              accel   lb               NONE     :291-296
     GA_CREATE_LISTENER    j              accel   NONE             NONE     :298-307
     GA_UPDATE_LISTENER    j              accel   listener         NONE     :313-321
     GA_CREATE_EG          j              accel   listener|NONE    lb       :322-331 (NONE: listener made by the preceding op)
     GA_UPDATE_EG          j              accel   eg               lb       :337-345
     GA_DELETE_CHAIN       0              accel   listener|NONE    eg|NONE  :254-288 (listener/eg only if exactly one exists)
     R53_CREATE            (j<<20)|k      zone    accel            NONE     route53.go:100-113 (TXT owner record, then A alias)
     R53_UPSERT_A          (j<<20)|k      zone    accel            record   route53.go:115-124
     R53_DELETE_RECORD     phase          zone    record           value    route53.go:132-165
   j = lbIngress index within the object, k = hostname index within the split route53-hostname annotation.
   Self-observation.  The reference mutates AWS between the iterations of its lbIngress / hostname loops and re-lists, so a later
   iteration of the SAME object sees what an earlier one did (ListGlobalAcceleratorByResource finds the accelerator created for
   lbIngress 0 and takes the update path for lbIngress 1, global_accelerator.go:133-157; updateEndpointGroup REPLACES the
   endpoint list, :987-1002; a hostname repeated in the route53 annotation finds the record just created, route53.go:92-124).
   The change set reproduces that against the frozen snapshot: from the second lbIngress that reaches the update/create stage
   on, an object's ops are what the reference would decide AFTER its own earlier ops — never a second GA_CREATE_CHAIN or a
   second R53_CREATE for the same name.  Such ops name resources that do not exist yet with GAR_PENDING:
     GA_UPDATE_ACCEL  a0 = PENDING          the accelerator of this object's earlier GA_CREATE_CHAIN
     GA_UPDATE_EG     a0 = PENDING | accel, a1 = PENDING   the endpoint group made by this object's earlier GA_CREATE_CHAIN /
                                                           GA_CREATE_LISTENER+GA_CREATE_EG / GA_CREATE_EG for that accelerator
     R53_UPSERT_A     a2 = PENDING          the A record of this object's earlier R53_CREATE for the same hostname string
   (User tags that overwrite the managed / owner / cluster tag with another value make an accelerator invisible to the list
   call once written: every later lbIngress then creates again, as the reference would.)
   R53_DELETE_RECORD: phase 0 = owned alias set (FindOwneredARecordSets), a2 = first value row of that zone
   whose value is the owner value and whose record has the alias set's name; phase 1 = owner metadata set
   (findOwneredMetadataRecordSets), a2 = the matching value row (one op per matching value, as the reference
   appends the set once per matching value). */
typedef enum {
  GAR_OP_GA_CREATE_CHAIN = 1,
  GAR_OP_GA_UPDATE_ACCEL = 2,
  GAR_OP_GA_CREATE_LISTENER = 3,
  GAR_OP_GA_UPDATE_LISTENER = 4,
  GAR_OP_GA_CREATE_EG = 5,
  GAR_OP_GA_UPDATE_EG = 6,
  GAR_OP_GA_DELETE_CHAIN = 7,
  GAR_OP_R53_CREATE = 8,
  GAR_OP_R53_UPSERT_A = 9,
  GAR_OP_R53_DELETE_RECORD = 10
} gar_opcode;

enum { GAR_CTRL_GA = 0, GAR_CTRL_R53 = 1 };

/* One op = 6 little-endian u32 words. */
typedef struct gar_op {
  uint32_t head; /* bits 0..7 gar_opcode, bits 8..15 GAR_CTRL_*, bits 16..23 GAR_KIND_* of obj (0 for orphans) */
  uint32_t obj;  /* object row, GAR_NONE for orphan ops */
  uint32_t sub;  /* see table above */
  uint32_t a0, a1, a2;
} gar_op;
#define GAR_OP_HEAD(op, ctrl, kind) ((uint32_t)(op) | ((uint32_t)(ctrl) << 8) | ((uint32_t)(kind) << 16))
#define GAR_R53_SUB(j, k) (((uint32_t)(j) << 20) | (uint32_t)(k))

/* Section order of `ops` (canonical; see DESIGN.md "Change-set order"):
     [0] GA ops of cached objects, by object row, then reference statement order
     [1] GA orphan deletes (owner tag of this cluster, no such object in the cache), by accelerator row
     [2] R53 ops of cached objects, by object row, then reference statement order
     [3] R53 orphan deletes, by (zone, phase, record row, value row) */
enum { GAR_SEC_GA_OBJ = 0, GAR_SEC_GA_ORPHAN = 1, GAR_SEC_R53_OBJ = 2, GAR_SEC_R53_ORPHAN = 3, GAR_N_SECTIONS = 4 };

/* Per-object derived desired state (what the create/update calls are fed; global_accelerator.go:214-225,503-557) */
enum {
  GAR_DV_PROTO_UDP = 1u << 0,      /* listenerForService protocol: last tcp/udp port wins (:503-515) */
  GAR_DV_IP_PRESERVE = 1u << 1,    /* client-ip-preservation annotation == "true" (:225) */
  GAR_DV_IPV4 = 1u << 2,           /* ip-address-type annotation in {"ipv4","IPV4"} (:686-695) */
  GAR_DV_PORTS_FROM_ANN = 1u << 3, /* Ingress carries alb.ingress.kubernetes.io/listen-ports: desired ports are
                                      dports[dport_begin[i]..], not port_number[] (:526-542) */
  GAR_DV_GA_ELIGIBLE = 1u << 4,    /* wasLoadBalancerService / wasALBIngress */
  GAR_DV_GA_MANAGED = 1u << 5,     /* hasManagedAnnotation (controller.go:250-253) */
  GAR_DV_R53_ELIGIBLE = 1u << 6,   /* route53 controller filter (route53/controller.go:87-148) */
  GAR_DV_R53_ANNOTATED = 1u << 7   /* hasHostnameAnnotation (route53/controller.go:243-246) */
};

/* gar_tok_code — result of DetectCloudProvider + GetLBNameFromHostname for one lbIngress hostname */
typedef enum {
  GAR_TOK_ALB_INTERNAL = 0,
  GAR_TOK_ALB_PUBLIC = 1,
  GAR_TOK_NLB = 2,
  GAR_TOK_NOT_AWS = 3,          /* DetectCloudProvider error -> `continue` (service.go:88-92) */
  GAR_TOK_PANIC = 4,            /* < 2 labels */
  GAR_TOK_ERR_NOT_ELB = 5,
  GAR_TOK_ERR_INTERNAL_ALB = 6,
  GAR_TOK_ERR_PUBLIC_ALB = 7,
  GAR_TOK_ERR_NLB = 8
} gar_tok_code;

typedef struct gar_changeset {
  uint32_t n_objects;
  const uint32_t *status_ga;   /* [n_objects] */
  const uint32_t *status_r53;  /* [n_objects] */
  const uint32_t *derived;     /* [n_objects] GAR_DV_* */
  uint64_t n_ops;
  const gar_op *ops;           /* [n_ops] */
  uint64_t section_begin[GAR_N_SECTIONS + 1];
  /* hostname tokeniser results, one per lbIngress row (name/region are refs into gar_objects.slab) */
  uint32_t n_lbi;
  const uint8_t *tok_code;     /* [n_lbi] gar_tok_code */
  const gar_str *tok_name;     /* [n_lbi] */
  const gar_str *tok_region;   /* [n_lbi] */
  /* desired port lists parsed from the listen-ports annotation (objects with GAR_DV_PORTS_FROM_ANN) */
  const uint32_t *dport_begin; /* [n_objects+1] */
  uint64_t n_dports;
  const int32_t *dports;       /* [n_dports] */
  /* sharded mode only (NULL otherwise): global object row of each local object row; ops then carry global rows */
  const uint32_t *obj_gid;     /* [n_objects] */
  /* timings of this diff, CUDA events on the engine's stream */
  float ms_h2d;                /* snapshot upload (measured at gar_snapshot_load) */
  float ms_kernels;            /* first kernel .. last kernel */
  float ms_d2h;                /* result download */
  uint32_t kernel_launches;    /* kernels launched by this diff */
  void *opaque;                /* engine-private; do not touch */
} gar_changeset;

typedef struct gar_engine gar_engine;

/* ---------------------------------------------------------------- entry points */

/* Create an engine bound to one CUDA device.  Fails with GAR_E_NO_DEVICE when there is no sm_100 GPU. */
int gar_engine_create(const gar_config *cfg, gar_engine **out);
void gar_engine_destroy(gar_engine *e);

/* Validate and copy a snapshot to the device (replaces any previous snapshot).
   Stands for: lister.List() on the two informers + the paginated AWS lists the per-object path issues
   (global_accelerator.go:624-652,789-813,885-907; route53.go:199-214,317-333; load_balancer.go:13-30). */
int gar_snapshot_load(gar_engine *e, const gar_objects *desired, const gar_actual *actual);

/* Same, for buffers that already live in device memory of the engine's device (all pointers in the two
   structs are device pointers, the structs themselves are host memory).  No copy is made: the caller keeps
   the buffers alive until the next load or gar_engine_destroy.  Table validation is skipped. */
int gar_snapshot_attach_device(gar_engine *e, const gar_objects *desired, const gar_actual *actual);

/* Compute the complete change set for both controllers against the loaded snapshot and copy it to host.
   Stands for: one processCreateOrUpdate / processDelete per key (globalaccelerator/service.go:28-126,
   ingress.go:29-130, route53/service.go:29-111, ingress.go:20-104) evaluated against the frozen snapshot. */
int gar_diff(gar_engine *e, gar_changeset *out);

/* Device-resident variant: runs the kernels only and leaves the result on the device.  Only the counts
   (n_ops, section_begin, n_dports) and timings of `out` are filled; array pointers are DEVICE pointers
   valid until the next diff/load on this engine. */
int gar_diff_device(gar_engine *e, gar_changeset *out);

/* Incremental mode (SURVEY.md §8 row f4): the decisions of a batch of work-queue keys against the loaded snapshot.
   `rows` are the object rows whose keys fired (informer add/update events, globalaccelerator/controller.go:91-111);
   `deleted_*` are keys that are no longer in the cache (delete events, :113-173): kind + "ns/name".
   Stands for: ProcessNextWorkItem once per key (pkg/reconcile/reconcile.go:26-42) -> processCreateOrUpdate for the
   rows, processDelete for the deleted keys.  The snapshot's digests and hash indexes are built on the first diff after
   a load and reused by every later gar_diff / gar_diff_keys until the next load.
   Result layout: n_objects = n_rows; status_ga[k], status_r53[k], derived[k] belong to rows[k]; object-section ops
   follow the order of `rows` and carry the real object row in `obj`; the orphan sections hold the cleanup ops of the
   deleted keys in the order given (per key: processDelete order, i.e. accelerators in list order / per zone alias
   sets then owner metadata sets); they carry obj = GAR_NONE.  tok_* and dports are not produced (n_lbi = 0,
   n_dports = 0). */
typedef struct gar_keyset {
  uint32_t n_rows;
  const uint32_t *rows;            /* [n_rows] object rows, each < n_objects */
  uint32_t n_deleted;
  const uint8_t *deleted_kind;     /* [n_deleted] GAR_KIND_* */
  const char *const *deleted_key;  /* [n_deleted] NUL-terminated "ns/name" */
} gar_keyset;
int gar_diff_keys(gar_engine *e, const gar_keyset *keys, gar_changeset *out);

/* ---------------------------------------------------------------- EndpointGroupBinding set-diff (SURVEY.md §8 row f3)
   The third controller's decisions (pkg/controller/endpointgroupbinding/reconcile.go:20-217): finalizer handling and the
   set difference between the load balancers of the referenced Service/Ingress and status.endpointIds.  Evaluated against
   the loaded snapshot (object cache, tokenised lbIngress hostnames, listed load balancers). */
enum { GAR_EGB_REF_NONE = 0, GAR_EGB_REF_SERVICE = 1, GAR_EGB_REF_INGRESS = 2 };
enum {
  GAR_EGB_DELETING = 1u << 0,       /* metadata.deletionTimestamp != nil (reconcile.go:27) */
  GAR_EGB_HAS_FINALIZERS = 1u << 1, /* len(metadata.finalizers) != 0 (:30) */
  GAR_EGB_OBSERVED = 1u << 2        /* status.observedGeneration == metadata.generation (:148) */
};
typedef struct gar_bindings {
  uint32_t n_bindings;
  const uint8_t *egb_flags;        /* GAR_EGB_* */
  const uint8_t *egb_ref_kind;     /* GAR_EGB_REF_*: spec.serviceRef / spec.ingressRef (:219-252) */
  const gar_str *egb_ref_key;      /* "<binding namespace>/<ref name>": the lister key of the referenced object */
  const gar_str *egb_eg_arn;       /* spec.endpointGroupArn */
  const uint32_t *egb_ep_begin;    /* [n_bindings+1] -> ep_id: status.endpointIds[] in order */
  uint32_t n_endpoint_ids;
  const gar_str *ep_id;
  uint32_t n_known_egs;            /* endpoint groups for which DescribeEndpointGroup succeeds (global_accelerator.go:867-876) */
  const gar_str *known_eg_arn;
  const uint8_t *slab;
  uint64_t slab_len;
} gar_bindings;

/* EGB ops (ctrl = GAR_CTRL_EGB, obj = binding row):
     EGB_ADD_FINALIZER      -            reconcileCreate  (:98-110)
     EGB_REMOVE_FINALIZER   -            reconcileDelete  (:36-47, :53-66)
     EGB_REMOVE_ENDPOINT    a0 = ep_id row                 RemoveLBFromEdnpointGroup (:80, :161)
     EGB_ADD_ENDPOINT       a0 = lb row                    AddLBToEndpointGroup (:172)
     EGB_UPDATE_WEIGHT      a0 = lb row                    UpdateEndpointWeight (:190)
     EGB_UPDATE_STATUS      -                              UpdateStatus (:87-90, :197-200)
   Go map iteration order (the `arns` map, :119,:139,:189) is unspecified; the canonical order here is first occurrence
   among the referenced object's lbIngress hostnames.  Statuses: GAR_ST_OK, GAR_ST_ERR_RETRY (GAR_D_*),
   GAR_ST_REQUEUE_30S (LB not active, global_accelerator.go:579-582), GAR_ST_REQUEUE_1S (:96), GAR_ST_PANIC (nil regional
   client when endpoints must be removed but the reference has no hostnames, :160; slice bounds in the delete loop, :84). */
enum { GAR_OP_EGB_ADD_FINALIZER = 11, GAR_OP_EGB_REMOVE_FINALIZER = 12, GAR_OP_EGB_REMOVE_ENDPOINT = 13, GAR_OP_EGB_ADD_ENDPOINT = 14,
       GAR_OP_EGB_UPDATE_WEIGHT = 15, GAR_OP_EGB_UPDATE_STATUS = 16 };
enum { GAR_CTRL_EGB = 2 };
enum { GAR_ST_REQUEUE_1S = 8 };
enum { GAR_D_REF_NOT_FOUND = 12, GAR_D_EG_NOT_FOUND = 13 };

/* Result: n_objects = n_bindings, status_ga[] holds the binding statuses, ops the EGB ops in binding order (one section);
   status_r53 / derived / tok_* / dports are not produced. */
int gar_bindings_diff(gar_engine *e, const gar_bindings *bindings, gar_changeset *out);

/* ---------------------------------------------------------------- sharded mode (SURVEY.md §8 row e, BASELINE configs[3])

   ONE cluster too large (or too slow) for one GPU, spread over n_ranks engines (one process per GPU).  Every rank loads
   (gar_snapshot_load) a SLICE: contiguous ranges of the object list and of each AWS list, in rank order (rank r holds
   global rows [base_r, base_r + n_r) of every table; nested rows travel with their parent), with these two rules:
     - the zone table (zone_name, zone_rec_begin) is complete and identical on every rank; a rank holds the record sets of
       whole zones only (other zones have empty record ranges), zone ranges ascending with the rank;
     - *_base give the global row of the slice's first row of each table.
   Both rules are checked on the device (a fingerprint of the zone table travels in the meta rows); a violation makes
   gar_shard_unpack return GAR_E_INVALID on the ranks that can see it — the host must propagate that to the other ranks
   before their next collective (shard.py does it with one all-reduce).
   Rows are then re-homed by key hash on the device in two exchanges the HOST performs between the calls below (the data
   path is torch.distributed all_to_all_single over NCCL in ranks.py, or any all-to-all):

     for round in 1, 2:
       gar_shard_route(e, &shard, round, meta, send_bytes)    meta[n_ranks][GAR_SHARD_META_WORDS]: row r describes the
                                                              blob for rank r; send_bytes[r] its size (multiple of 16)
       exchange the meta rows (all-to-all of GAR_SHARD_META_WORDS u64 per peer)
       gar_shard_pack(e, send)                                send: device buffer of sum(send_bytes), blobs back to back
       exchange the blobs (all-to-all, sizes from gar_shard_blob_bytes(received meta row))
       gar_shard_unpack(e, round, recv, recv_meta)            recv: the received blobs back to back, in rank order, with
                                                              32 readable bytes behind them.  The string bytes are NOT
                                                              copied: the sub-snapshot's strings live in BOTH rounds' receive
                                                              buffers, which must stay alive and unchanged until the last
                                                              diff of this exchange (the next gar_shard_route(.., 1) or
                                                              gar_snapshot_load ends their use; between that route call
                                                              and its second unpack gar_diff returns GAR_E_STATE)
   Round 1 moves every row to the shard its own key hashes to and one probe per lbIngress hostname to the "directory"
   shard of that hostname; round 2 returns the load balancer / by-hostname accelerators each probe resolves to.  After the
   second unpack the engine holds a self-contained sub-snapshot: gar_diff / gar_diff_device work as usual, n_objects is
   the number of objects homed here, obj_gid[] gives their global rows, ops carry GLOBAL rows and keep the canonical order
   within the shard (merge shards by (section, key row) for the cluster-wide order).  Stands for nothing in the reference
   (it has one process and no batch); semantics = gar_diff over the concatenated slices, which the tests check bit for bit. */
#define GAR_SHARD_MAX_RANKS 8
#define GAR_SHARD_META_WORDS 40
typedef struct gar_shard {
  uint32_t rank, n_ranks;
  uint32_t obj_base, lb_base, acc_base, lis_base, eg_base, rec_base, val_base;
} gar_shard;
int gar_shard_route(gar_engine *e, const gar_shard *shard, int round, uint64_t *meta, uint64_t *send_bytes);
int gar_shard_pack(gar_engine *e, void *send);
int gar_shard_unpack(gar_engine *e, int round, const void *recv, const uint64_t *recv_meta);
uint64_t gar_shard_blob_bytes(const uint64_t *meta_row);

/* Peer-memory exchange (one process per GPU on one NVLink / NVSwitch node): no collective on the data path.  Every rank maps the
   RECEIVE arenas of the other GPUs through CUDA IPC; gar_shard_pack_peers packs the rank's own blob in place and the others into a
   local stage from which a copy kernel on a high-priority stream pushes them into the peers' arenas over NVLink (16-byte coalesced
   stores), level group by level group while the later levels are still being packed (transfer and partitioning overlap).
   On 8 B200s this beat copy engines, pack kernels storing straight into the mapped arenas, and bulk stores from shared memory
   (DESIGN.md §6).  Per round:

     gar_shard_route(e, &shard, round, meta, send_bytes)
     all-gather the meta rows                                  -> all_meta[s][d] = row of source s for destination d
     gar_shard_arena(e, round, need, &ptr, handle, &cap)       need = sum over s of gar_shard_blob_bytes(all_meta[s][rank]);
                                                               (re)allocates this rank's arena of the round and exports it
     all-gather the handles; gar_shard_open_peers(e, round, handles)     (mappings are cached: re-opened only when a handle changed)
     gar_shard_pack_peers(e, round, all_meta)                  source s writes its blob for d at offset sum_{s' < s} blob bytes(s', d)
     barrier over the ranks (every pack has completed)         gar_shard_pack_peers has synchronised its own stream before returning
     gar_shard_unpack(e, round, ptr, column `rank` of all_meta)

   Same result as the send-buffer + all-to-all path above (tests compare both with the unsharded diff).  The host still moves
   the few hundred bytes of meta rows and handles (any all-gather); the bulk data never touches a collective library. */
#define GAR_SHARD_HANDLE_BYTES 96
int gar_shard_arena(gar_engine *e, int round, uint64_t need_bytes, void **arena, uint8_t *handle /* [GAR_SHARD_HANDLE_BYTES] */, uint64_t *capacity);
int gar_shard_open_peers(gar_engine *e, int round, const uint8_t *handles /* [n_ranks][GAR_SHARD_HANDLE_BYTES], rank order */);
int gar_shard_pack_peers(gar_engine *e, int round, const uint64_t *all_meta /* [n_ranks][n_ranks][GAR_SHARD_META_WORDS] */);

void gar_changeset_free(gar_engine *e, gar_changeset *cs);

const char *gar_last_error(const gar_engine *e); /* never NULL; valid until the next call on e */
const char *gar_version(void);

/* Bytes the diff must touch at least once: input slabs + fixed-width columns (each once)
   + 4 B per (controller, object) status + 24 B per op.  The roofline numerator (DESIGN.md §Measurement). */
uint64_t gar_algorithmic_bytes(const gar_engine *e, const gar_changeset *cs);

/* Per-stage device times of the last gar_diff / gar_diff_device (engine created with GAR_FLAG_STAGE_TIMING).
   Stages launched several times (index builds) are summed under one name.  Returns the number of stages. */
typedef struct gar_stage_timing {
  const char *name; /* static string */
  float ms;         /* CUDA-event time on the engine's stream */
  uint32_t launches;
  uint64_t bytes;   /* algorithmic bytes of the stage (DESIGN.md "Per-kernel byte model"), 0 if not modelled */
} gar_stage_timing;
uint32_t gar_last_stage_timings(gar_engine *e, gar_stage_timing *out, uint32_t cap);

/* Work counters of the last gar_diff / gar_diff_device / gar_diff_keys: exact sizes of the intermediate relations, for the
   per-kernel byte models of the roofline report (bench.py).  out[GAR_CTR_*]; returns the number of counters written. */
enum {
  GAR_CTR_R53_PAIRS = 0,   /* (object, route53 hostname) pairs evaluated by the r53_pairs stage (route53.go:84-124 loop bodies) */
  GAR_CTR_DPORTS = 1,      /* ports parsed from listen-ports annotations */
  GAR_CTR_N = 2
};
uint32_t gar_last_counters(gar_engine *e, uint64_t *out, uint32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* GARECON_H */
