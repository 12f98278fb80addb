#!/usr/bin/env python
"""bench.py — objects reconciled / second on synthetic informer caches (BASELINE.json metric).

One "step" = one complete diff (both controllers, every object, orphans) over one synthetic snapshot.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA engine
  python bench.py --impl reference [...]                          # CPU arm: the oracle port of the Go reference

Workload (config.workload): BASELINE.json configs[2] — 10^6 Service+Ingress, every object carrying a
multi-hostname route53 annotation, ~10^6 accelerators / 2*10^6 record sets on the AWS side (the config the
metric "objects reconciled/sec at 10^6" is quoted on; it fits one B200).  N > 1 is weak scaling: every rank
diffs its own 10^6-object cluster (independent clusters shard with no data-path collective; DESIGN.md §Multi-GPU).

JSON keys beyond the base contract:
  value      device-resident: snapshot already in HBM, timed region = K x gar_diff_device (all kernels + the two
             4-byte count read-backs the pipeline needs), wall clock between device synchronisations, max over ranks
  e2e        same metric through the C ABI with HOST (pinned) buffers: K x (gar_snapshot_load + gar_diff), i.e. H2D of
             every table + kernels + D2H of the whole change set inside the timed region
  roofline   HBM roofline of the dominant kernel and of the whole pipeline (CUDA events on the engine's stream)
  cpu_baseline  the oracle (C++ port of the reference decision functions, indexed, all host threads) on a bounded sample
The Go reference itself is NOT timed: there is no Go toolchain in this image (BASELINE.md §2).
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

METRIC = "objects reconciled/sec at 10^6 Service+Ingress; change-set bit-exact vs Go ref"
UNIT = "objects/s"


def _peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0: float, t1: float) -> dict:
        sel = [r for (t, r) in self.rows if t0 <= t <= t1 and len(r) >= 9] or [r for (_, r) in self.rows if len(r) >= 9]
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(r[1]) for r in sel if r[1].replace(".", "").isdigit()]
        smax = [float(r[2]) for r in sel if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in sel:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons), "samples": len(sel)}


def _table_arrays(abi, o, a):
    """(ctypes pointer, element count, element size) for every input array, in struct order."""
    n = o.n_objects
    out = [(o.obj_kind, n, 1), (o.obj_spec_type, n, 1), (o.obj_flags, n, 1), (o.obj_ns, n, 8), (o.obj_name, n, 8), (o.obj_ingress_class, n, 8),
           (o.obj_ann_begin, n + 1, 4), (o.obj_lbi_begin, n + 1, 4), (o.obj_port_begin, n + 1, 4), (o.ann_key, o.n_ann, 8), (o.ann_val, o.n_ann, 8),
           (o.lbi_hostname, o.n_lbi, 8), (o.port_number, o.n_ports, 4), (o.port_proto, o.n_ports, 8), (o.slab, o.slab_len + 32, 1),
           (a.lb_region, a.n_lbs, 8), (a.lb_name, a.n_lbs, 8), (a.lb_dns, a.n_lbs, 8), (a.lb_arn, a.n_lbs, 8), (a.lb_state, a.n_lbs, 1),
           (a.acc_name, a.n_accels, 8), (a.acc_dns, a.n_accels, 8), (a.acc_enabled, a.n_accels, 1),
           (a.acc_tag_begin, a.n_accels + 1, 4), (a.acc_lis_begin, a.n_accels + 1, 4), (a.tag_key, a.n_tags, 8), (a.tag_val, a.n_tags, 8),
           (a.lis_proto, a.n_listeners, 1), (a.lis_pr_begin, a.n_listeners + 1, 4), (a.lis_eg_begin, a.n_listeners + 1, 4),
           (a.pr_from, a.n_port_ranges, 4), (a.eg_ep_begin, a.n_egs + 1, 4), (a.ep_id, a.n_endpoints, 8),
           (a.zone_name, a.n_zones, 8), (a.zone_rec_begin, a.n_zones + 1, 4), (a.rec_name, a.n_records, 8),
           (a.rec_type, a.n_records, 1), (a.rec_has_alias, a.n_records, 1), (a.rec_alias_dns, a.n_records, 8), (a.rec_val_begin, a.n_records + 1, 4),
           (a.val_value, a.n_values, 8), (a.slab, a.slab_len + 32, 1)]
    return out


def _np_col(ptr, n, dtype):
    import numpy as np
    n = int(n)
    if n == 0:
        return np.zeros(0, dtype=dtype)
    addr = C.cast(ptr, C.c_void_p).value
    return np.frombuffer((C.c_char * (n * np.dtype(dtype).itemsize)).from_address(addr), dtype=dtype, count=n)


def _key_is(col, slab_ptr, slab_len, literal: bytes):
    """Boolean mask over a gar_str column: rows whose string equals `literal` (length AND bytes, chunked so that the gathered
    candidates stay small)."""
    import numpy as np
    lens = (col >> np.uint64(40)).astype(np.int64)
    mask = lens == len(literal)
    cand = np.flatnonzero(mask)
    if not len(cand) or not literal:
        return mask
    slab = _np_col(slab_ptr, slab_len, np.uint8)
    want = np.frombuffer(literal, dtype=np.uint8)
    offs = (col[cand] & np.uint64((1 << 40) - 1)).astype(np.int64)
    step = 1 << 16
    for b in range(0, len(cand), step):
        o = offs[b:b + step]
        same = (slab[o[:, None] + np.arange(len(literal))[None, :]] == want[None, :]).all(axis=1)
        mask[cand[b:b + step][~same]] = False
    return mask


DUMP_VALUES_MAX = 1 << 19  # per dumped array: 4 MB of float64, so the eleven arrays stay under DUMP_BYTES_MAX
DUMP_BYTES_MAX = 64 << 20
DUMP_SEED = 0


class _DeviceBytes:
    """`nbytes` bytes at a device address, readable by torch through the CUDA array interface."""

    def __init__(self, addr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (addr, False), "version": 2}


def device_changeset(torch, cs):
    """Host copies of the arrays of a device-resident gar_changeset (what gar_diff_device hands its caller), under the names of
    abi.ChangeSet.  Call it before the next diff or load on the engine: the pointers are only valid until then."""
    import numpy as np
    from types import SimpleNamespace
    abi = importlib.import_module("aws-global-accelerator-controller_b200.abi")

    def pull(ptr, n, dtype):
        nbytes = int(n) * np.dtype(dtype).itemsize
        if nbytes == 0:
            return np.zeros(0, dtype=dtype)
        raw = torch.as_tensor(_DeviceBytes(C.cast(ptr, C.c_void_p).value, nbytes), device="cuda").cpu().numpy()
        return raw.view(dtype)

    n, nlbi = int(cs.n_objects), int(cs.n_lbi)
    return SimpleNamespace(
        status_ga=pull(cs.status_ga, n, np.uint32), status_r53=pull(cs.status_r53, n, np.uint32), derived=pull(cs.derived, n, np.uint32),
        ops=pull(cs.ops, cs.n_ops, abi.OP_DTYPE), section_begin=np.array(list(cs.section_begin), dtype=np.uint64),
        tok_code=pull(cs.tok_code, nlbi, np.uint8), tok_name=pull(cs.tok_name, nlbi, np.uint64), tok_region=pull(cs.tok_region, nlbi, np.uint64),
        dport_begin=pull(cs.dport_begin, n + 1, np.uint32), dports=pull(cs.dports, cs.n_dports, np.int32))


def dump_outputs(cs, out_dir, max_values: int = DUMP_VALUES_MAX) -> dict:
    """Write the change set `cs` (numpy arrays named as in abi.ChangeSet) as float64 `out_dir/<name>.npy`, every value exact:
    ops as (n_ops, 6) rows of head, obj, sub, a0, a1, a2; the gar_str columns tok_name / tok_region as (n_lbi, 2) rows of slab
    offset, length.  An array with more than `max_values` values keeps a sample of its rows: the same ascending row indices for
    the same row count (fixed seed), so two runs on the same inputs are compared row for row.  `counts` holds the full sizes
    (objects, ops, lbIngress hostnames, derived ports).  Returns {name: rows written}."""
    import numpy as np
    str_cols = lambda v: np.stack([v & np.uint64((1 << 40) - 1), v >> np.uint64(40)], axis=1)
    arrays = {
        "status_ga": cs.status_ga, "status_r53": cs.status_r53, "derived": cs.derived,
        "ops": np.stack([cs.ops[f] for f in cs.ops.dtype.names], axis=1),
        "section_begin": cs.section_begin, "tok_code": cs.tok_code, "tok_name": str_cols(cs.tok_name), "tok_region": str_cols(cs.tok_region),
        "dport_begin": cs.dport_begin, "dports": cs.dports,
        "counts": np.array([len(cs.status_ga), len(cs.ops), len(cs.tok_code), len(cs.dports)]),
    }
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    written, total = {}, 0
    for name, a in arrays.items():
        rows = max(1, max_values // max(1, int(np.prod(a.shape[1:]))))
        if len(a) > rows:
            a = a[np.sort(np.random.default_rng(DUMP_SEED).choice(len(a), rows, replace=False))]
        a = a.astype(np.float64)
        total += a.nbytes
        if total > DUMP_BYTES_MAX:
            raise ValueError(f"--dump-outputs: more than {DUMP_BYTES_MAX >> 20} MB of outputs")
        np.save(out_dir / f"{name}.npy", a)
        written[name] = len(a)
    return written


TAG_OWNER_KEY, TAG_THOST_KEY = b"aws-global-accelerator-owner", b"aws-global-accelerator-target-hostname"
TAG_MANAGED_KEY, TAG_CLUSTER_KEY = b"aws-global-accelerator-controller-managed", b"aws-global-accelerator-cluster"
ANN_R53_KEY = b"aws-global-accelerator-controller.h3poteto.dev/route53-hostname"


def kernel_byte_models(o, a, n_ops_ga_obj: int, n_pairs: int, frac_ga: float):
    """Algorithmic bytes of the two decide kernels (DESIGN.md "Per-kernel byte model"): the unique input bytes each must
    read at least once + what it must write.  Index/digest structures it reads are counted (they are its inputs);
    re-reads, sector padding and scratch are not."""
    import numpy as np
    L = lambda ptr, n: int((_np_col(ptr, n, np.uint64) >> np.uint64(40)).sum())
    n = o.n_objects
    key_bytes = L(o.obj_ns, n) + L(o.obj_name, n) + n
    host_bytes = L(o.lbi_hostname, o.n_lbi)
    lb_strings = L(a.lb_region, a.n_lbs) + L(a.lb_name, a.n_lbs) + L(a.lb_dns, a.n_lbs) + L(a.lb_arn, a.n_lbs)
    tkc = _np_col(a.tag_key, a.n_tags, np.uint64)
    tv = _np_col(a.tag_val, a.n_tags, np.uint64) >> np.uint64(40)
    is_owner, is_thost = _key_is(tkc, a.slab, a.slab_len, TAG_OWNER_KEY), _key_is(tkc, a.slab, a.slab_len, TAG_THOST_KEY)
    is_managed, is_cluster = _key_is(tkc, a.slab, a.slab_len, TAG_MANAGED_KEY), _key_is(tkc, a.slab, a.slab_len, TAG_CLUSTER_KEY)
    thost_bytes = int(tv[is_thost].sum())
    owner_bytes = int(tv[is_owner].sum())
    acc_strings = L(a.acc_name, a.n_accels) + thost_bytes + owner_bytes + L(a.ep_id, a.n_endpoints)
    ga = frac_ga * (host_bytes + 17 * o.n_lbi + lb_strings + (32 + 16) * a.n_lbs + acc_strings + (32 + 64) * a.n_accels) \
        + n * (4 + 8 + 16 + 8 + 1) + key_bytes + 4 * o.n_ports * frac_ga + n * 8 + 24 * n_ops_ga_obj
    nrec, nval = a.n_records, a.n_values
    val_bytes = L(a.val_value, nval)
    name_bytes_per_rec = L(a.rec_name, nrec) / max(nrec, 1)
    alias_bytes_per_rec = L(a.rec_alias_dns, nrec) / max(int(_np_col(a.rec_has_alias, nrec, np.uint8).sum()), 1)
    acc_dns_per = L(a.acc_dns, a.n_accels) / max(a.n_accels, 1)
    zone_name_per = L(a.zone_name, a.n_zones) / max(a.n_zones, 1)
    # per pair: hostname piece, pair row, zone entry + name, the object's value entries (32 B each, ~1 per pair) with the
    # owner-key bytes of the in-zone one, its record name, the value->alias link, the alias DNS name, the accelerator DNS name
    is_r53 = _key_is(_np_col(o.ann_key, o.n_ann, np.uint64), o.slab, o.slab_len, ANN_R53_KEY)
    av = _np_col(o.ann_val, o.n_ann, np.uint64) >> np.uint64(40)
    ann_r53 = int(av[is_r53].sum())
    r53 = ann_r53 + n_pairs * ((4 + 8) + (1 + 4 + 4) + 32 + zone_name_per + 32 + key_bytes / max(n, 1) + name_bytes_per_rec + 16 + alias_bytes_per_rec + acc_dns_per + 8 + 8 + 1 + 16)
    models = {"ga_objects": int(ga), "r53_pairs": int(r53)}
    # ---- the other stages: input bytes each must read once + output bytes it writes (same rules: no re-reads, no scratch)
    ann_key_refs = 8 * o.n_ann
    known_key_bytes = 1024  # interned annotation keys: a handful of distinct strings
    models["classify_objects"] = int(n * (3 + 3 * 8 + 3 * 4) + ann_key_refs + 8 * o.n_ann + known_key_bytes + key_bytes + n * (4 + 8 + 4 * 8 + 4))
    models["tokenise_hostnames"] = int(host_bytes + 8 * o.n_lbi + 17 * o.n_lbi)
    sys_tag_bytes = int(tv[is_owner | is_thost | is_managed | is_cluster].sum())
    models["digest_accelerators"] = int(a.n_accels * (2 * 4 + 2 * 8 + 1) + 16 * a.n_tags + sys_tag_bytes + a.n_listeners * (1 + 8) + 4 * a.n_port_ranges
                                        + 4 * a.n_egs + 8 * a.n_endpoints + a.n_accels * (64 + 5 * 8 + 2 * 8 + 4))
    name_bytes = L(a.rec_name, nrec)
    models["prepare_records"] = int(name_bytes + nrec * (8 + 4) + val_bytes + 8 * nval + nrec * (4 + 8) + nval * (4 + 1 + 8 + 8))
    n_owner_vals = nval  # generator: every TXT value is an owner value (orphans and foreign clusters included)
    models["value_joins"] = int(n_owner_vals * ((1 + 8 + 8 + 4) + (8 + 32 + 2 * name_bytes_per_rec) + (8 + 32 + 2 * key_bytes / max(n, 1)) + 16 + 1))
    # index build (one pass over every index): per row its key hash and payload columns read once (~28 B), one 32-byte entry written,
    # one 4-byte cursor touched, + the scanned bucket array read once for the multi-entry list
    idx_rows_total = a.n_lbs + 2 * a.n_accels + a.n_zones + nval + nrec + n
    models["idx_place"] = int(idx_rows_total * (28 + 32 + 4) + 4 * idx_rows_total)
    models["idx_order"] = int(idx_rows_total * 0.25 * (4 + 2.5 * 32 * 2))  # ~a quarter of the buckets hold 2-3 entries: read + written back
    models["hash_load_balancers"] = int(L(a.lb_region, a.n_lbs) + L(a.lb_name, a.n_lbs) + a.n_lbs * (16 + 8 + 4))
    n_annotated = int(is_r53.sum())
    models["r53_prepare"] = int(n * (4 + 8 + 1) + host_bytes + n_annotated * (32 + 8 + acc_dns_per) + ann_r53 + n * (1 + 4 + 8 + 4))
    models["r53_objects"] = int(n * (1 + 4 + 4 + 4) + n_pairs * (1 + 4 + 4) + n * 8)
    models["r53_fill_pairs"] = int(n * (4 + 8) + ann_r53 + n_pairs * (4 + 8))
    return models


def _pin_host_tables(torch, abi, o, a):
    """cudaHostRegister every generator-owned array so the e2e arm copies from pinned memory.  -> (bytes, [addresses])"""
    rt = torch.cuda.cudart()
    pinned, addrs = 0, []
    for ptr, cnt, sz in _table_arrays(abi, o, a):
        nbytes = int(cnt) * sz
        addr = C.cast(ptr, C.c_void_p).value
        if not addr or nbytes == 0:
            continue
        rc = rt.cudaHostRegister(addr, nbytes, 0)
        if int(rc) == 0:
            pinned += nbytes
            addrs.append(addr)
    return pinned, addrs


def _unpin(torch, addrs):
    rt = torch.cuda.cudart()
    for a in addrs:
        rt.cudaHostUnregister(a)


CPU_TUNED, CPU_LITERAL = 2, 1  # oracle modes: the tuned host-core baseline (flat indexes, tag digests, thread pool) / the literal indexed port


def _cpu_arm(ob, snap, threads_list, reps=1, mode=CPU_TUNED):
    """objects/s of a CPU mode of the oracle on `snap` for each thread count: {threads: objects/s}"""
    n = int(snap.objects.n_objects)
    out = {}
    for t in threads_list:
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            ob.diff_raw(snap.objects, snap.actual, snap.cluster.encode(), mode, t)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        out[int(t)] = n / best
    return out


def _thread_ladder(cores):
    return sorted({t for t in (1, 8, 32, 64, 128, cores) if t <= cores})


def _best_threads(scaling):
    """The thread count the CPU arm is reported at: the fastest of the ladder (on an SMT box all hardware threads can be slower
    than half of them; the baseline is the best the host can do, not a fixed count)."""
    return max(scaling, key=lambda t: scaling[t])


def run_reference(args, rank, world):
    """CPU arm: the oracle (port of the reference's decision functions; indexed mode, all host threads) on the SAME workload
    as the GPU arm: the full --objects cluster of --config, same generator seed and slab layout."""
    if rank != 0:
        return
    import __graft_entry__ as ge
    ge.build_synth()
    ge.build_oracle()
    synth = importlib.import_module("aws-global-accelerator-controller_b200.synth")
    ob = importlib.import_module("oracle.binding")
    cores = os.cpu_count() or 1
    n = args.objects if args.cpu_sample <= 0 else min(args.cpu_sample, args.objects)
    cfg = synth.preset(args.config, n)
    cfg.layout = 1 if args.layout == "column" else 0
    snap = synth.SynthSnapshot(cfg)
    cl = snap.cluster.encode()
    scaling = _cpu_arm(ob, snap, _thread_ladder(cores))  # one untimed pass per thread count: warm-up and the choice of the count
    best_t = _best_threads(scaling)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ob.diff_raw(snap.objects, snap.actual, cl, CPU_TUNED, best_t)
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    scaling[best_t] = value
    literal = _cpu_arm(ob, snap, [cores], mode=CPU_LITERAL)[cores]
    cores_used = best_t
    sample = (f"the whole workload: config {args.config} generator at {n} objects (seed {int(cfg.seed)}, {args.layout}-major slabs); oracle mode 2 "
              f"(tuned: flat hash indexes, tag digests, thread pool; bit-identical to the literal port, tests/test_synth_configs.py), {best_t} threads "
              f"= the fastest of the ladder in `scaling` on this host ({cores} hardware threads)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32 (bytes and indices)",
        "data": "synthetic", "config": {"workload": _workload_name(args.config, args.objects), "sample_objects": n, "same_config": n == args.objects,
                                        "slab_layout": args.layout, "seed": int(cfg.seed)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores_used, "kind": "port", "sample": sample,
                         "scaling": {str(k): round(v, 1) for k, v in sorted(scaling.items())},
                         "literal_port": {"value": literal, "cores": cores, "what": "oracle mode 1: the function-by-function restatement over unordered_map indexes"}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "Go reference not timed (no Go toolchain in this image); CPU baseline is a C++ restatement of the reference's decision functions; "
                "with N > 1 GPUs the GPU arm diffs N clusters of this size, this arm one (rank 0 only, per the bench contract)",
    }
    print(json.dumps(line), flush=True)


_WORKLOADS = {1: "100 Services type LoadBalancer (plumbing)", 2: "Service+Ingress vs mocked AWS lists (hash-join diff)",
              3: "Service+Ingress with multi-hostname route53 annotation", 4: "cfg2 u cfg3 mix (the sharded 10^7 cluster)",
              5: "adversarial: 90% colliding hostnames + 64-port listeners"}


def _workload_name(config, objects):
    return f"BASELINE configs[{config - 1}]: {objects} objects, {_WORKLOADS.get(config, '')}"


def _cache_note(bytes_per_gpu):
    """how the timed iterations avoid a warm L2 (126 MB): inputs larger than L2, or say that they are not"""
    if bytes_per_gpu > 2 * 126e6:
        return f"inputs ({bytes_per_gpu / 1e6:.0f} MB per GPU) larger than L2 (126 MB); no flush needed"
    return f"inputs ({bytes_per_gpu / 1e6:.0f} MB per GPU) do NOT exceed L2 (126 MB): an L2-sized scratch buffer is rewritten between timed steps"


SHARD_CHUNKS = 16  # the sharded cluster is always generated as 16 chunks, whatever the number of GPUs


def sharded_measure(args, R, rank, world, local_rank, n_total, cfg_id, steps, warmup, with_single=True, detail=True):
    """BASELINE configs[3]: ONE cluster of n_total objects; every GPU starts with an arbitrary slice of each list (objects /
    accelerators / load balancers of different generator chunks on each rank), rows are re-homed by key hash (one all-to-all
    of rows + a small answer exchange), every GPU diffs its self-contained shard.  Returns the record (rank 0) or None.

    Parity inside the run (outside the timed regions): the additive canonical checksum (shard.canonical_checksum) of the
    per-shard HOST change sets, summed over the ranks, must equal the checksum of the single-GPU diff of the same cluster."""
    import torch
    pkg = importlib.import_module("aws-global-accelerator-controller_b200")
    synth = importlib.import_module("aws-global-accelerator-controller_b200.synth")
    shard = importlib.import_module("aws-global-accelerator-controller_b200.shard")
    dev = torch.device("cuda", local_rank)
    cores = os.cpu_count() or 8
    gen_threads = max(2, min(48, cores // max(world, 1)))
    layout = 1 if args.layout == "column" else 0
    n_chunks = SHARD_CHUNKS if (SHARD_CHUNKS % world == 0 and n_total % SHARD_CHUNKS == 0) else world
    n_total -= n_total % n_chunks
    tg = time.perf_counter()
    o_cols, a_cols = synth.cluster_slices(cfg_id, n_total, world, ranks=[rank], layout=layout, n_chunks=n_chunks, threads=gen_threads)[0]
    snap = pkg.tables.from_columns(o_cols, a_cols)
    gen_s = time.perf_counter() - tg
    counts = R.gather_counts([len(o_cols["obj_kind"]), len(a_cols["lb_state"]), len(a_cols["acc_enabled"]), len(a_cols["lis_proto"]),
                              len(a_cols["eg_ep_begin"]) - 1, len(a_cols["rec_type"]), len(a_cols["val_value"]), snap.input_bytes()])
    base = [sum(c[k] for c in counts[:rank]) for k in range(7)]
    sh = pkg.abi.GarShard(rank, world, *base)
    h2d_bytes = snap.input_bytes()
    _, pinned_addrs = _pin_host_tables(torch, pkg.abi, snap.objects, snap.actual)
    eng = pkg.Engine(cluster_name="default", device=local_rank)
    Exchange = shard.PeerExchange if args.exchange == "p2p" else shard.DistExchange
    ex = Exchange(eng, sh, dev)
    sampler = ClockSampler(local_rank)
    sampler.start()

    def step():
        ex.run()
        return eng.diff_device()

    eng.load(snap)
    launches = 0
    for _ in range(warmup):
        cs = step()
    R.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        cs = step()
        launches += cs.kernel_launches
    R.barrier()
    t1 = time.perf_counter()
    dt_dev = R.max_over_ranks(t1 - t0)
    clocks = sampler.summary(t0, t1)
    homed = int(cs.n_objects)
    sent = ex.bytes_sent
    # end to end: host slice in (H2D), host change set out (D2H), every step
    for _ in range(2):
        eng.load(snap)
        ex.run()
        eng.diff_raw()
    R.barrier()
    t2 = time.perf_counter()
    for _ in range(steps):
        eng.load(snap)
        ex.run()
        eng.diff_raw()
    R.barrier()
    t3 = time.perf_counter()
    dt_e2e = R.max_over_ranks(t3 - t2)
    sampler.stop()
    # parity: this shard's host change set -> additive checksum, summed over the ranks
    part = eng.diff()
    n_ops = len(part.ops)
    ck = shard.canonical_checksum(part)
    del part
    lo, hi = ck["sum"] & 0xFFFFFFFF, ck["sum"] >> 32
    allck = R.gather_counts([lo, hi, ck["n_objects"], ck["n_ops"]] + ck["sections"])
    # phase breakdown (separate pass, synchronised between phases; not part of the timed numbers above)
    ex.timing, ex.phase_ms = True, {}
    phases = {}
    for _ in range(3):
        ex.run()
        torch.cuda.synchronize()
        ta = time.perf_counter()
        eng.diff_device()
        torch.cuda.synchronize()
        phases["diff"] = phases.get("diff", 0.0) + (time.perf_counter() - ta) * 1e3 / 3
    for k, v in ex.phase_ms.items():
        phases[k] = v / 3
    ex.timing = False
    eng.close()
    stage_acc = {}
    if detail:  # per-kernel CUDA-event times of one whole sharded step (engine with GAR_FLAG_STAGE_TIMING; separate pass)
        peng = pkg.Engine(cluster_name="default", device=local_rank, stage_timing=True)
        peng.load(snap)
        pex = Exchange(peng, sh, dev)
        for it in range(4):
            pex.run()
            peng.diff_device()
            if it == 0:
                continue
            for name, ms, nl in peng.stage_timings():
                e = stage_acc.setdefault(name, [0.0, 0])
                e[0] += ms / 3
                e[1] += nl
        peng.close()
    ex.keep.clear()
    _unpin(torch, pinned_addrs)
    del ex, snap, o_cols, a_cols
    torch.cuda.empty_cache()
    allc = R.gather_counts([homed, n_ops, sent, int(sum(phases.values()) * 1000)] + [int(phases[k] * 1000) for k in sorted(phases)])
    # ---- the same cluster on ONE GPU (rank 0): the strong-scaling denominator and the parity arbiter
    single = None
    if with_single and rank == 0:
        tg = time.perf_counter()
        slices = synth.cluster_slices(cfg_id, n_total, world, layout=layout, n_chunks=n_chunks, threads=min(48, cores))
        union = pkg.tables.concat_slices(slices)
        del slices
        gen1_s = time.perf_counter() - tg
        _, addrs1 = _pin_host_tables(torch, pkg.abi, union.objects, union.actual)
        with pkg.Engine(cluster_name="default", device=local_rank, reprepare=True) as e1:
            e1.load(union)
            whole = e1.diff()
            ck1 = shard.canonical_checksum(whole)
            del whole
            for _ in range(warmup):
                e1.diff_device()
            torch.cuda.synchronize()
            ta = time.perf_counter()
            for _ in range(steps):
                e1.diff_device()
            torch.cuda.synchronize()
            dt1 = time.perf_counter() - ta
            for _ in range(1):
                e1.load(union)
                e1.diff_raw()
            tb = time.perf_counter()
            for _ in range(max(1, steps // 2)):
                e1.load(union)
                e1.diff_raw()
            dt1e = (time.perf_counter() - tb) / max(1, steps // 2)
        single = {"value": n_total * steps / dt1, "ms_per_step": dt1 / steps * 1e3, "e2e_value": n_total / dt1e, "e2e_ms_per_step": dt1e * 1e3,
                  "checksum": ck1, "input_bytes": union.input_bytes(), "generate_s": round(gen1_s, 1)}
        _unpin(torch, addrs1)
        del union
    R.barrier()
    if rank != 0:
        return None
    peak, peak_src = _peaks()
    in_bytes = sum(c[7] for c in counts)
    b_alg = in_bytes + 8 * n_total + 24 * sum(c[1] for c in allc)
    value = n_total * steps / dt_dev
    achieved = b_alg / (dt_dev / steps) / 1e9
    merged = {"sum": sum((c[0] | (c[1] << 32)) for c in allck) & 0xFFFFFFFFFFFFFFFF, "n_objects": sum(c[2] for c in allck), "n_ops": sum(c[3] for c in allck),
              "sections": [sum(c[4 + k] for c in allck) for k in range(4)]}
    ph_max = {k: max(c[4 + i] for c in allc) / 1000 for i, k in enumerate(sorted(phases))}
    exch_ms = sum(v for k, v in ph_max.items() if k != "diff")
    sent_max = max(c[2] for c in allc)
    # where the bytes cross NVLink: the all-to-all of the send-buffer path, the pack kernels themselves with peer memory
    xfer = ["pack1", "pack2"] if args.exchange == "p2p" else ["transfer1", "transfer2"]
    rec = {
        "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": dt_dev / steps * 1e3, "scaling": "strong",
        "config": {"workload": f"BASELINE configs[3]: ONE cluster of {n_total} Service+Ingress (generator preset {cfg_id}, {n_chunks} chunks, {args.layout}-major slabs) "
                               f"cut into {world} slices (objects / accelerators / load balancers of different chunk groups on each rank), re-homed by key hash",
                   "objects_total": n_total,
                   "parallelism": f"key-hash shards x{world}: " + ("pack kernels store the rows straight into the peers' receive arenas over NVLink (CUDA IPC), " if args.exchange == "p2p"
                                                                   else "pack -> NCCL all_to_all_single -> unpack, ") + "rows + answer round, then local diff",
                   "exchange": args.exchange,
                   "cache": _cache_note(h2d_bytes), "homed_objects_per_rank": [c[0] for c in allc], "ops_per_rank": [c[1] for c in allc],
                   "algorithmic_bytes": b_alg, "generate_s": round(gen_s, 1)},
        "e2e": {"value": n_total * steps / dt_e2e, "unit": UNIT, "h2d_bytes_per_step": in_bytes,
                "d2h_bytes_per_step": 12 * n_total + 24 * sum(c[1] for c in allc), "ms_per_step": dt_e2e / steps * 1e3},
        "gpu_launches": launches, "clocks": clocks,
        "bytes_sent": {"per_rank": [c[2] for c in allc], "max": sent_max,
                       "nvlink_gbs_per_direction_in_transfer": round(sent_max / max(sum(ph_max.get(k, 0) for k in xfer), 1e-9) / 1e6, 1),
                       "transfer_phases": xfer, "nvlink_peak_gbs_per_direction": 900.0, "nvlink_measured_peer_copy_gbs": 770.0},
        "roofline": {"bound": "hbm", "kernel": "whole sharded step (route, pack, exchange, merge, diff)", "achieved": achieved, "peak": peak * world,
                     "unit": "GB/s", "frac": achieved / (peak * world), "traffic": None, "peak_source": peak_src + f" x {world} GPUs"},
        "phases_ms_rank0": {k: round(v, 3) for k, v in phases.items()},
        "phases_ms_max_over_ranks": ph_max,
        "exchange_ms_max_over_ranks": round(exch_ms, 3),
        "stages_ms_rank0": {k: round(v[0], 4) for k, v in sorted(stage_acc.items(), key=lambda kv: -kv[1][0])},
        "checksum": merged,
    }
    if single is not None:
        rec["single_gpu_value"] = single["value"]
        rec["single_gpu"] = single
        rec["strong_scaling_speedup"] = value / single["value"]
        rec["strong_scaling_efficiency"] = value / single["value"] / world
        rec["e2e_speedup"] = rec["e2e"]["value"] / single["e2e_value"]
        rec["checksum_equal"] = merged == single["checksum"]
    return rec


def run_sharded(args, rank, world, local_rank):
    """`--mode sharded`: the sharded step as the bench line's own metric (the default invocation under torchrun reports it as
    the `sharded` record of the replicas line instead)."""
    import torch
    import __graft_entry__ as ge
    ranks_mod = importlib.import_module("aws-global-accelerator-controller_b200.ranks")
    dev = torch.device("cuda", local_rank)
    R = ranks_mod.Ranks(backend="nccl", device=dev)
    if world == 1 and not R.dist.is_initialized():  # single GPU: a 1-rank group keeps the code path identical
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29577")
        R.dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
        R.owns_group = True
    if rank == 0:
        ge.ensure_built()
    R.barrier()
    cfg_id = 4 if args.config == 3 else args.config  # default workload of this mode: configs[3] = generator preset 4
    rec = sharded_measure(args, R, rank, world, local_rank, args.objects, cfg_id, args.steps, args.warmup, with_single=not args.no_single)
    if rank == 0:
        line = {"metric": METRIC, "higher_is_better": True, "vs_baseline": None, "dtype": "u8/u32 (bytes and indices)", "data": "synthetic"}
        line.update(rec)
        print(json.dumps(line), flush=True)
    R.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="garecon", choices=["garecon", "reference"])
    ap.add_argument("--config", type=int, default=3, help="BASELINE.json configs index (1-based): 3 = 10^6 multi-hostname route53")
    ap.add_argument("--objects", type=int, default=1_000_000)
    ap.add_argument("--cpu-sample", type=int, default=0, help="objects of the CPU baseline's workload; 0 = the whole workload (same config as the GPU arm)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle comparison of the timed workload's change set")
    ap.add_argument("--layout", default="column", choices=["row", "column"],
                    help="where the packer puts strings inside the slabs: column = every string column contiguous (what host/packer.hpp writes; "
                         "default), row = row-major by parent object (9 %% slower: DESIGN.md §3).  Results do not depend on it.")
    ap.add_argument("--mode", default="replicas", choices=["replicas", "sharded"],
                    help="replicas: one independent cluster per GPU (weak scaling, no collective); with N > 1 GPUs the line also carries a "
                         "`sharded` record: ONE 10^7-object cluster re-homed by key hash across the GPUs (BASELINE configs[3], strong scaling, "
                         "checksum-compared with the same cluster on one GPU).  sharded: only that, as the line's own metric")
    ap.add_argument("--sharded-objects", type=int, default=10_000_000, help="size of the cluster of the `sharded` record")
    ap.add_argument("--sharded-steps", type=int, default=5)
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the sharded record")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="sharded mode data path: p2p = pack kernels store straight into the other GPUs' receive arenas (CUDA IPC peer memory); "
                         "nccl = pack into a send buffer, torch.distributed all_to_all_single, unpack")
    ap.add_argument("--no-single", action="store_true", help="sharded: skip the single-GPU run of the same cluster (no checksum comparison)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the change set of the last timed step (rank 0) as DIR/<name>.npy, float64, "
                         "at most 64 MB (large arrays as a fixed-seed sample of their rows; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "garecon" or args.mode != "replicas"):
        ap.error("--dump-outputs writes the change set of the replicas step of this repo's engine (--impl garecon --mode replicas)")
    args.warmup = max(args.warmup, 3) if args.impl == "garecon" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    if args.mode == "sharded":
        run_sharded(args, rank, world, local_rank)
        return
    import __graft_entry__ as ge
    pkg = importlib.import_module("aws-global-accelerator-controller_b200")
    synth = importlib.import_module("aws-global-accelerator-controller_b200.synth")
    ranks_mod = importlib.import_module("aws-global-accelerator-controller_b200.ranks")
    binding = ranks_mod.NumaBinding(local_rank)  # host tables are first-touched (and later pinned) on the GPU's own NUMA node
    numa = binding.node
    R = ranks_mod.Ranks(backend="nccl", device=torch.device("cuda", local_rank))
    if rank == 0:
        ge.ensure_built()
    R.barrier()
    abi = pkg.abi
    barrier, max_over_ranks = R.barrier, R.max_over_ranks

    # ---- workload: one synthetic cluster per rank (different seed per rank)
    cfg = synth.preset(args.config, args.objects)
    cfg.seed = ranks_mod.rank_seed(cfg.seed, rank)
    cfg.layout = 1 if args.layout == "column" else 0
    snap = synth.SynthSnapshot(cfg)
    o, a = snap.objects, snap.actual
    h2d_bytes = sum(int(c) * s for (_, c, s) in _table_arrays(abi, o, a))
    pinned_bytes, pinned_addrs = _pin_host_tables(torch, abi, o, a)
    binding.release()
    # inputs that fit in L2 would make every timed step after the first an L2-warm re-read: rewrite an L2-sized buffer between steps
    flush = h2d_bytes <= 2 * 126e6
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}") if flush else None

    # reprepare=True: every timed step runs the COMPLETE pipeline (digests, indexes, decide, placement); without it the
    # engine would reuse the prepared snapshot after the first diff, which is the incremental-mode optimisation, not the metric
    eng = pkg.Engine(cluster_name=snap.cluster, device=local_rank, reprepare=True)
    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- device-resident arm ("value")
    eng.load(snap)
    launches = 0
    for _ in range(args.warmup):
        cs = eng.diff_device()
    barrier()
    t0 = time.perf_counter()
    ms_kernels = 0.0
    t_flush = 0.0
    for _ in range(args.steps):
        if flush:
            tf = time.perf_counter()
            flush_buf.fill_(1)
            torch.cuda.synchronize()
            t_flush += time.perf_counter() - tf
        cs = eng.diff_device()
        ms_kernels += cs.ms_kernels
        launches += cs.kernel_launches
    barrier()
    t1 = time.perf_counter()
    dt_dev = max_over_ranks(t1 - t0 - t_flush)
    if args.dump_outputs and rank == 0:  # before the e2e arm reloads the engine, which ends the device pointers of `cs`
        dump_outputs(device_changeset(torch, cs), args.dump_outputs)
    b_alg = eng.algorithmic_bytes(cs)
    n_ops = int(cs.n_ops)
    n_pairs = eng.counters().get("r53_pairs", 0)
    d2h_bytes = 4 * 3 * o.n_objects + 24 * n_ops + 17 * o.n_lbi + 4 * (o.n_objects + 1) + 4 * int(cs.n_dports)
    clocks = sampler.summary(t0, t1)

    # ---- end-to-end arm: host tables in, host change set out, every step
    for _ in range(2):
        eng.load(snap)
        full = eng.diff_raw()
    barrier()
    t2 = time.perf_counter()
    e2e_parts = {"ms_h2d": 0.0, "ms_kernels": 0.0, "ms_d2h": 0.0}
    for _ in range(args.steps):
        eng.load(snap)
        full = eng.diff_raw()  # C-ABI calls only: gar_snapshot_load + gar_diff (host change set in pinned memory) + free
        e2e_parts["ms_h2d"] += full["ms_h2d"] / args.steps
        e2e_parts["ms_kernels"] += full["ms_kernels"] / args.steps
        e2e_parts["ms_d2h"] += full["ms_d2h"] / args.steps
    barrier()
    t3 = time.perf_counter()
    dt_e2e_local = t3 - t2
    dt_e2e = max_over_ranks(dt_e2e_local)
    e2e_per_rank = R.gather_counts([int(dt_e2e_local / args.steps * 1e6), int(e2e_parts["ms_h2d"] * 1e3), int(e2e_parts["ms_kernels"] * 1e3),
                                    int(e2e_parts["ms_d2h"] * 1e3), -1 if numa is None else numa])
    sampler.stop()

    # ---- parity gate (rank 0, outside the timed regions): the change set of the timed workload, bit for bit against the oracle
    parity = {"checked": False}
    hcs = None
    if rank == 0:
        eng.load(snap)
        hcs = eng.diff()
        if not args.no_parity:
            ob = importlib.import_module("oracle.binding")
            tp = time.perf_counter()
            want = ob.diff(snap, snap.cluster, mode=1, threads=os.cpu_count() or 4)
            bad = hcs.diff(want)
            parity = {"checked": True, "equal": not bad, "oracle_objects": int(o.n_objects), "oracle": "oracle/oracle.cpp indexed mode (C++ port of the Go decision functions)",
                      "arrays_compared": list(hcs.ARRAYS), "n_ops": int(len(want.ops)), "seconds": round(time.perf_counter() - tp, 2)}
            if bad:
                parity["mismatch"] = {"arrays": bad, "first": hcs.describe_first_mismatch(want)}
            del want
    eng.close()

    # ---- roofline pass (separate engine with per-stage CUDA events; not part of the timed numbers above)
    peak, peak_src = _peaks()
    stages = []
    if rank == 0:
        peng = pkg.Engine(cluster_name=snap.cluster, device=local_rank, stage_timing=True, reprepare=True)
        peng.load(snap)
        acc = {}
        reps = max(3, min(args.steps, 10))
        for it in range(reps + 2):
            if flush:
                flush_buf.fill_(1)
                torch.cuda.synchronize()
            peng.diff_device()
            if it < 2:
                continue
            for name, ms, nl in peng.stage_timings():
                e = acc.setdefault(name, [0.0, 0])
                e[0] += ms
                e[1] += nl
        stages = sorted(((name, v[0] / reps, v[1] // reps) for name, v in acc.items()), key=lambda x: -x[1])
        pipeline_ms = sum(s[1] for s in stages)
        top = stages[0]
        peng.close()
    total_objects = args.objects * world

    line = None
    if rank == 0:
        value = total_objects * args.steps / dt_dev
        e2e_value = total_objects * args.steps / dt_e2e
        pipe_achieved = b_alg / (pipeline_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u32 (bytes and indices)", "data": "synthetic",
            "config": {"workload": _workload_name(args.config, args.objects) + f" per GPU; {a.n_accels} accelerators, {a.n_records} record sets, {a.n_lbs} load balancers",
                       "slab_layout": args.layout, "objects_per_gpu": args.objects, "parallelism": f"replicas x{world} (independent clusters, no collective)",
                       "cache": _cache_note(h2d_bytes), "seed": int(cfg.seed),
                       "n_ops": n_ops, "r53_pairs": n_pairs, "algorithmic_bytes": b_alg, "bytes_per_object": b_alg / args.objects},
            "parity": parity,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes, "ms_per_step": dt_e2e / args.steps * 1e3,
                    "pinned_host_bytes": pinned_bytes, **{k: round(v, 3) for k, v in e2e_parts.items()},
                    "per_rank": [{"ms_per_step": c[0] / 1e3, "ms_h2d": c[1] / 1e3, "ms_kernels": c[2] / 1e3, "ms_d2h": c[3] / 1e3, "numa_node": c[4]} for c in e2e_per_rank]},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": top[0], "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
                         "peak_source": peak_src, "kernel_ms": top[1], "kernel_share": top[1] / pipeline_ms,
                         "pipeline": {"achieved": pipe_achieved, "frac": pipe_achieved / peak, "ms": pipeline_ms, "bytes": b_alg},
                         "stages_ms": {s[0]: round(s[1], 4) for s in stages}},
            "kernel_ms_per_step_cuda_events": ms_kernels / args.steps,
        }
        # the dominant kernel's own byte model (DESIGN.md "Per-kernel byte model"); the pipeline figure is the headline
        frac_ga = float(((hcs.status_ga & 0xFF) > 2).sum() + ((hcs.status_ga & 0xFF) == 1).sum()) / max(args.objects, 1)
        sb = [int(x) for x in hcs.section_begin]
        models = kernel_byte_models(o, a, sb[1] - sb[0], n_pairs, frac_ga)
        traffic, traffic_src = {}, None
        for tp in (REPO / "profiles" / "r02_ncu_traffic.json", REPO / "profiles" / "r01_ncu_traffic.json"):
            if tp.exists() and args.config == 3 and args.objects == 1_000_000:  # the capture is of this exact workload
                traffic = json.loads(tp.read_text()).get("dram_bytes_per_launch", {})
                traffic_src = f"profiles/{tp.name} (ncu --set full, same workload)"
                break
        # every stage with a byte model: its own achieved GB/s and fraction of the HBM roofline (CUDA-event stage times)
        line["roofline"]["kernels"] = {name: {"ms": round(ms, 4), "bytes": models[name], "achieved_gbs": round(models[name] / (ms * 1e-3) / 1e9, 1),
                                              "frac": round(models[name] / (ms * 1e-3) / 1e9 / peak, 4)}
                                       for name, ms, _ in stages if name in models and ms > 0}
        kb = models.get(top[0])
        if kb:
            line["roofline"]["achieved"] = kb / (top[1] * 1e-3) / 1e9
            line["roofline"]["frac"] = line["roofline"]["achieved"] / peak
            line["roofline"]["kernel_bytes"] = kb
            line["roofline"]["traffic"] = traffic.get(top[0])
            line["roofline"]["traffic_source"] = traffic_src if top[0] in traffic else None
        else:
            line["roofline"]["achieved"] = pipe_achieved
            line["roofline"]["frac"] = pipe_achieved / peak
        # incremental mode (not the headline): batches of 1 % dirty keys against the prepared, resident snapshot,
        # through gar_diff_keys with host buffers (rows in, statuses + ops out)
        try:
            import random as _random
            ieng = pkg.Engine(cluster_name=snap.cluster, device=local_rank)
            ieng.load(snap)
            rng = _random.Random(7)
            nb = max(1, args.objects // 100)
            batches = [abi.make_keyset(sorted(rng.sample(range(args.objects), nb))) for _ in range(8)]
            cs_k = abi.GarChangeset()
            for ks in batches[:2]:
                ieng._check(ieng.lib.gar_diff_keys(ieng._h, C.byref(ks), C.byref(cs_k)))
                ieng.lib.gar_changeset_free(ieng._h, C.byref(cs_k))
            torch.cuda.synchronize()
            tk = time.perf_counter()
            for ks in batches[2:]:
                ieng._check(ieng.lib.gar_diff_keys(ieng._h, C.byref(ks), C.byref(cs_k)))
                ieng.lib.gar_changeset_free(ieng._h, C.byref(cs_k))
            dtk = (time.perf_counter() - tk) / len(batches[2:])
            ieng.close()
            line["incremental"] = {"batch_keys": nb, "ms_per_batch": dtk * 1e3, "keys_per_s": nb / dtk,
                                   "note": "gar_diff_keys on a prepared snapshot (digests + indexes resident), host rows in / host change set out"}
        except Exception as ex:  # never let the side measurement break the contract line
            line["incremental"] = {"error": str(ex)[:200]}
        if not args.no_cpu_baseline:
            ob = importlib.import_module("oracle.binding")
            cores = os.cpu_count() or 1
            if args.cpu_sample and args.cpu_sample < args.objects:
                csnap = synth.generate(args.config, args.cpu_sample)
                same = False
            else:
                csnap, same = snap, True
            cn = int(csnap.objects.n_objects)
            scaling = _cpu_arm(ob, csnap, _thread_ladder(cores), reps=1)
            literal = _cpu_arm(ob, csnap, sorted({1, cores}), mode=CPU_LITERAL)
            # the reference's own algorithm (per object: linear scan of all accelerators / all records, O(N*A)): timed at
            # two small sizes to show the quadratic growth; it is the bit-exactness arbiter, not a fair batch baseline
            faithful = []
            for fn in (1000, 4000):
                fs = synth.generate(args.config, fn)
                tf = time.perf_counter()
                ob.diff_raw(fs.objects, fs.actual, fs.cluster.encode(), 0, 1)
                fdt = time.perf_counter() - tf
                faithful.append({"objects": fn, "seconds": round(fdt, 3), "objects_per_s": round(fn / fdt, 1)})
            line["cpu_faithful"] = {"kind": "port", "cores": 1, "runs": faithful,
                                    "note": "literal per-object linear scans as in the reference (quadratic); indexed multi-thread figure is cpu_baseline"}
            best_t = _best_threads(scaling)
            line["cpu_baseline"] = {"value": scaling[best_t], "unit": UNIT, "cores": best_t, "kind": "port", "same_config": same,
                                    "scaling": {str(k): round(v, 1) for k, v in sorted(scaling.items())},
                                    "literal_port": {"scaling": {str(k): round(v, 1) for k, v in sorted(literal.items())},
                                                     "what": "oracle mode 1: the function-by-function restatement over unordered_map indexes (the parity arbiter)"},
                                    "sample": f"{'the timed workload itself' if same else 'a sample'}: config {args.config} generator at {cn} objects, oracle mode 2 (tuned: flat "
                                              f"hash indexes, tag digests, thread pool; bit-identical to the literal port), {best_t} threads = the fastest of the ladder in `scaling` ({cores} hardware threads); "
                                              f"Go reference not timed (no toolchain)"}
    _unpin(torch, pinned_addrs)
    del snap, o, a, hcs, flush_buf
    torch.cuda.empty_cache()
    # ---- N > 1: BASELINE configs[3] — ONE 10^7-object cluster sharded by key hash across the GPUs (same JSON line)
    if world > 1 and not args.no_sharded:
        try:
            rec = sharded_measure(args, R, rank, world, local_rank, args.sharded_objects, 4, args.sharded_steps, 3, with_single=not args.no_single, detail=False)
        except Exception as ex:  # the replicas line must survive a failure here; every rank raises together (DistExchange agrees on errors)
            rec = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
        if rank == 0:
            line["sharded"] = rec
    if rank == 0:
        print(json.dumps(line), flush=True)
    R.close()


if __name__ == "__main__":
    main()
