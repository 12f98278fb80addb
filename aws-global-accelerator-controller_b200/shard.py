"""Sharded mode: ONE cluster spread over several engines (include/garecon.h "sharded mode", csrc/gar_shard.h).

The engine plans, packs and merges; moving the blobs between ranks is the host's job and lives here:

  exchange_dist   one process per GPU, torch.distributed all_to_all_single (NCCL over NVLink on the GPU box, gloo in the
                  CPU tests): one all-to-all of the meta rows + one of the blobs per round
  exchange_local  every rank's engine in this process, buffers in host memory (the hostsim test tier)

`merge_changesets` puts per-shard results back into the cluster-wide canonical order so they can be compared with the
unsharded diff bit for bit.
"""
from __future__ import annotations

import numpy as np

from . import abi

NONE = 0xFFFFFFFF


# ------------------------------------------------------------------ slicing a dict model (tests, small cases)

def slice_model(objects: list[dict], actual: dict, n_ranks: int):
    """Cut a tables.pack() model into n_ranks slices the way a packer would: contiguous ranges of every list, whole
    zones per rank, the zone table replicated.  -> [(objects_r, actual_r, GarShard)], rank order."""
    def cuts(n):
        return [n * r // n_ranks for r in range(n_ranks + 1)]

    accs, lbs, zones = actual.get("accelerators", []), actual.get("lbs", []), actual.get("zones", [])
    co, ca, cl, cz = cuts(len(objects)), cuts(len(accs)), cuts(len(lbs)), cuts(len(zones))
    out = []
    base = dict(obj=0, lb=0, acc=0, lis=0, eg=0, rec=0, val=0)
    for r in range(n_ranks):
        objs_r = objects[co[r]:co[r + 1]]
        accs_r = accs[ca[r]:ca[r + 1]]
        lbs_r = lbs[cl[r]:cl[r + 1]]
        zones_r = [dict(z, records=(z.get("records", []) if cz[r] <= i < cz[r + 1] else [])) for i, z in enumerate(zones)]
        sh = abi.GarShard(r, n_ranks, base["obj"], base["lb"], base["acc"], base["lis"], base["eg"], base["rec"], base["val"])
        out.append((objs_r, dict(accelerators=accs_r, lbs=lbs_r, zones=zones_r), sh))
        base["obj"] += len(objs_r)
        base["lb"] += len(lbs_r)
        base["acc"] += len(accs_r)
        for a in accs_r:
            base["lis"] += len(a.get("listeners", []))
            base["eg"] += sum(len(li.get("egs", [])) for li in a.get("listeners", []))
        for z in zones_r:
            base["rec"] += len(z["records"])
            base["val"] += sum(len(rec.get("values", [])) for rec in z["records"])
    return out


# ------------------------------------------------------------------ exchanges

def exchange_local(engines, shards, keep, device="cpu"):
    """Both rounds for engines that all live in this process: host-memory backends (device="cpu", the hostsim test tier) or
    several engines on one GPU (device="cuda:0").  `keep` collects the buffers that must outlive the call (the engines
    read the round-1 blobs again in round 2)."""
    import torch
    g = len(engines)
    for rnd in (1, 2):
        metas, sends = [], []
        for e, sh in zip(engines, shards):
            meta, nbytes = e.shard_route(sh, rnd)
            buf = torch.zeros(int(nbytes.sum()) + 64, dtype=torch.uint8, device=device)
            if str(device) != "cpu":
                torch.cuda.synchronize()  # the fill runs on torch's stream, the engine packs on its own: order them
            e.shard_pack(buf.data_ptr())
            metas.append(meta)
            sends.append((buf, np.concatenate([[0], np.cumsum(nbytes)]).astype(np.int64)))
        for d, e in enumerate(engines):
            recv_meta = np.stack([metas[s][d] for s in range(g)])
            parts = [sends[s][0][int(sends[s][1][d]):int(sends[s][1][d + 1])] for s in range(g)]
            recv = torch.cat(parts + [torch.zeros(64, dtype=torch.uint8, device=device)])
            if str(device) != "cpu":
                torch.cuda.synchronize()
            keep.append(recv)
            e.shard_unpack(rnd, recv.data_ptr(), recv_meta)


def exchange_local_peers(engines, shards):
    """Both rounds over peer memory for engines that all live in this process (hostsim: host arenas; several engines on one
    GPU: device arenas, no IPC needed): every engine's pack stores straight into the other engines' receive arenas."""
    g = len(engines)
    for rnd in (1, 2):
        metas = [e.shard_route(sh, rnd)[0] for e, sh in zip(engines, shards)]
        all_meta = np.stack(metas)  # [source][destination][words]
        arenas, handles = [], []
        for d, e in enumerate(engines):
            need = sum(e.blob_bytes(all_meta[s][d]) for s in range(g))
            ptr, h, _ = e.shard_arena(rnd, need)
            arenas.append(ptr)
            handles.append(h)
        handles = np.stack(handles)
        for e in engines:
            e.shard_open_peers(rnd, handles)
        for e in engines:
            e.shard_pack_peers(rnd, all_meta)
        for d, e in enumerate(engines):
            e.shard_unpack(rnd, arenas[d], np.ascontiguousarray(all_meta[:, d]))


_MAX_BLOB_BYTES = 1 << 40  # what a 40-bit string offset can address: a meta row that claims more is corrupt, not big


def _check_blob_sizes(sizes, what):
    """Sizes derived from meta rows another rank sent: refuse nonsense before it becomes an allocation or a collective."""
    for s, n in enumerate(sizes):
        if n < 0 or n % 16 or n >= _MAX_BLOB_BYTES:
            raise ValueError(f"sharded exchange: implausible blob size {n} in the meta row of rank {s} ({what})")


class DistExchange:
    """torch.distributed data path of one rank.  Buffers are torch uint8 tensors on `device` (cuda:N or cpu)."""

    def __init__(self, engine, shard, device):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.e, self.shard, self.device = engine, shard, device
        self.g = int(shard.n_ranks)
        self.keep = []
        self.bytes_sent = 0
        self.check_errors = True  # one tiny all-reduce after the calls that can fail on one rank only (route, unpack)
        self.timing = False       # True: every phase is bracketed by device synchronisations and accumulated in phase_ms
        self.phase_ms = {}

    def _timed(self, name, fn):
        if not self.timing:
            return fn()
        import time
        sync = self.torch.cuda.synchronize if str(self.device) != "cpu" else (lambda: None)
        sync()
        t0 = time.perf_counter()
        out = fn()
        sync()
        self.phase_ms[name] = self.phase_ms.get(name, 0.0) + (time.perf_counter() - t0) * 1e3
        return out

    def _agree(self, err):
        """All ranks learn whether any rank failed its last engine call (otherwise the healthy ones would wait forever in the
        next collective).  Raises on every rank."""
        torch, dist = self.torch, self.dist
        flag = torch.tensor([1 if err is not None else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if int(flag.item()):
            if err is not None:
                raise err
            raise RuntimeError("sharded exchange aborted: another rank reported an engine error")

    def _guard(self, fn):
        err, out = None, None
        try:
            out = fn()
        except Exception as ex:  # noqa: BLE001 - reported to every rank, then re-raised
            err = ex
        if self.check_errors:
            self._agree(err)
        elif err is not None:
            raise err
        return out

    def round(self, rnd: int):
        torch, dist = self.torch, self.dist
        meta, nbytes = self._timed(f"route{rnd}", lambda: self._guard(lambda: self.e.shard_route(self.shard, rnd)))
        # meta rows: a fixed-size all-to-all (int64 view of the uint64 words)
        m_out = torch.from_numpy(meta.view(np.int64)).to(self.device)
        m_in = torch.empty_like(m_out)
        self._timed(f"meta{rnd}", lambda: dist.all_to_all_single(m_in, m_out))
        recv_meta = m_in.cpu().numpy().view(np.uint64)
        in_sizes = [int(x) for x in nbytes]
        out_sizes = [self.e.blob_bytes(recv_meta[s]) for s in range(self.g)]
        self._guard(lambda: _check_blob_sizes(out_sizes, "received"))
        send = torch.empty(sum(in_sizes) + 64, dtype=torch.uint8, device=self.device)
        if str(self.device) != "cpu":
            torch.cuda.current_stream().synchronize()  # the allocation (and any fill) is on torch's stream, the engine packs on its own
        # a pack failure on one rank must not leave the others in the all-to-all
        self._timed(f"pack{rnd}", lambda: self._guard(lambda: self.e.shard_pack(send.data_ptr())))
        recv = torch.empty(sum(out_sizes) + 64, dtype=torch.uint8, device=self.device)
        self._timed(f"transfer{rnd}", lambda: dist.all_to_all_single(recv[:sum(out_sizes)], send[:sum(in_sizes)], output_split_sizes=out_sizes, input_split_sizes=in_sizes))
        if str(self.device) != "cpu":
            torch.cuda.current_stream().synchronize()  # the engine reads `recv` on its own stream
        self.keep.append(recv)
        self.bytes_sent += sum(in_sizes)
        self._timed(f"unpack{rnd}", lambda: self._guard(lambda: self.e.shard_unpack(rnd, recv.data_ptr(), recv_meta)))

    def run(self):
        """Both rounds; afterwards the engine holds this rank's home sub-snapshot (diff() works)."""
        self.keep.clear()
        self.bytes_sent = 0
        self.round(1)
        self.round(2)


# ------------------------------------------------------------------ putting shard results back together

_SECTION_KEY = {
    0: lambda ops: (ops["obj"],),
    1: lambda ops: (ops["a0"],),
    2: lambda ops: (ops["obj"],),
    3: lambda ops: (ops["a2"], ops["a1"], ops["sub"], ops["a0"]),  # np.lexsort: last key is the primary one
}


def merge_changesets(parts, n_objects: int):
    """Per-shard ChangeSets (global rows, shard-local canonical order) -> cluster-wide statuses and ops in the canonical
    order of include/garecon.h.  Returns dict(status_ga, status_r53, derived, ops, section_begin)."""
    st_ga = np.zeros(n_objects, dtype=np.uint32)
    st_r53 = np.zeros(n_objects, dtype=np.uint32)
    derived = np.zeros(n_objects, dtype=np.uint32)
    seen = np.zeros(n_objects, dtype=np.uint32)
    for cs in parts:
        g = cs.obj_gid
        st_ga[g] = cs.status_ga
        st_r53[g] = cs.status_r53
        derived[g] = cs.derived
        seen[g] += 1
    if not np.all(seen == 1):
        raise AssertionError("every object must be homed on exactly one shard")
    sections, begins = [], [0]
    for sec in range(4):
        chunks = [cs.ops[int(cs.section_begin[sec]):int(cs.section_begin[sec + 1])] for cs in parts]
        ops = np.concatenate(chunks) if chunks else np.zeros(0, dtype=abi.OP_DTYPE)
        if len(ops):
            order = np.lexsort(_SECTION_KEY[sec](ops)) if sec == 3 else np.argsort(_SECTION_KEY[sec](ops)[0], kind="stable")
            ops = ops[order]
        sections.append(ops)
        begins.append(begins[-1] + len(ops))
    return dict(status_ga=st_ga, status_r53=st_r53, derived=derived, ops=np.concatenate(sections) if sections else np.zeros(0, dtype=abi.OP_DTYPE),
                section_begin=np.array(begins, dtype=np.uint64))


# ------------------------------------------------------------------ merge-free parity: a checksum that adds over shards

_M1, _M2, _M3 = np.uint64(0x9E3779B185EBCA87), np.uint64(0xC2B2AE3D27D4EB4F), np.uint64(0x165667B19E3779F9)


def _mix(h, v):
    h = (h ^ (v.astype(np.uint64) * _M2)) * _M1
    return h ^ (h >> np.uint64(29))


def _run_index(key_cols, n):
    """position of every element inside its run of equal consecutive keys"""
    if n == 0:
        return np.zeros(0, dtype=np.uint64)
    change = np.zeros(n, dtype=bool)
    change[0] = True
    for k in key_cols:
        change[1:] |= k[1:] != k[:-1]
    idx = np.arange(n, dtype=np.int64)
    start = np.maximum.accumulate(np.where(change, idx, 0))
    return (idx - start).astype(np.uint64)


def canonical_checksum(cs) -> dict:
    """Order-aware checksum of a change set that ADDS over shards: the sum (mod 2^64) of the per-shard values of one cluster
    equals the value of the unsharded change set iff (up to hash collisions) the merged result is identical — every status
    word is hashed with its GLOBAL object row, every op with its section, its canonical key (object row / accelerator row /
    (zone, phase, record, value)) and its position among the ops of that key, which is exactly what `merge_changesets`
    reconstructs.  Works on a ChangeSet of a whole cluster (rows = 0..n) and of a shard (rows = obj_gid, ops carry global rows).
    Returns {"sum": int, "n_objects": int, "n_ops": int, "sections": [4 sizes]}; add the fields over the shards."""
    with np.errstate(over="ignore"):
        n = int(cs.n_objects)
        rows = (cs.obj_gid if getattr(cs, "obj_gid", None) is not None else np.arange(n, dtype=np.uint32)).astype(np.uint64)
        h = _mix(np.full(n, 0x51A7, dtype=np.uint64), rows)
        for col in (cs.status_ga, cs.status_r53, cs.derived):
            h = _mix(h, col)
        total = int(h.sum(dtype=np.uint64)) if n else 0
        sb = [int(x) for x in cs.section_begin]
        for sec in range(4):
            ops = cs.ops[sb[sec]:sb[sec + 1]]
            m = len(ops)
            if not m:
                continue
            keys = [ops["obj"]] if sec in (0, 2) else ([ops["a0"]] if sec == 1 else [ops["a0"], ops["sub"], ops["a1"], ops["a2"]])
            h = _mix(np.full(m, 0xC0DE + sec, dtype=np.uint64), _run_index(keys, m))
            for f in ("head", "obj", "sub", "a0", "a1", "a2"):
                h = _mix(h, ops[f])
            total = (total + int(h.sum(dtype=np.uint64))) & 0xFFFFFFFFFFFFFFFF
        return {"sum": total, "n_objects": n, "n_ops": int(len(cs.ops)), "sections": [sb[k + 1] - sb[k] for k in range(4)]}


def add_checksums(parts) -> dict:
    out = {"sum": 0, "n_objects": 0, "n_ops": 0, "sections": [0, 0, 0, 0]}
    for p in parts:
        out["sum"] = (out["sum"] + p["sum"]) & 0xFFFFFFFFFFFFFFFF
        out["n_objects"] += p["n_objects"]
        out["n_ops"] += p["n_ops"]
        out["sections"] = [a + b for a, b in zip(out["sections"], p["sections"])]
    return out


class PeerExchange(DistExchange):
    """One process per GPU on one NVLink node: no collective on the data path.  Every rank maps the other GPUs' receive arenas
    (CUDA IPC, include/garecon.h "Peer-memory exchange"); gar_shard_pack_peers packs and a push kernel copies the blobs
    into the peers' arenas while later levels still pack.  torch.distributed moves one small all-gather per round (meta rows +
    arena handle, 0.4 KB per rank) and provides the barrier after the packs."""

    def round(self, rnd: int):
        torch, dist = self.torch, self.dist
        g = self.g
        me = int(self.shard.rank)
        meta, nbytes = self._timed(f"route{rnd}", lambda: self._guard(lambda: self.e.shard_route(self.shard, rnd)))

        def gather():
            # the arena as it stands (capacities only grow, so after the first step it fits) rides along with the meta rows
            arena, handle, cap = self._guard(lambda: self.e.shard_arena(rnd, 0))
            row = np.concatenate([meta.view(np.uint8).reshape(-1), handle, np.array([cap], dtype=np.uint64).view(np.uint8)])
            out = torch.from_numpy(row).to(self.device)
            gathered = torch.empty(g * row.size, dtype=torch.uint8, device=self.device)
            dist.all_gather_into_tensor(gathered, out)
            gathered = gathered.cpu().numpy().reshape(g, row.size)
            all_meta = np.ascontiguousarray(gathered[:, :meta.nbytes]).view(np.uint64).reshape((g,) + meta.shape)  # [source][destination][words]
            handles = np.ascontiguousarray(gathered[:, meta.nbytes:meta.nbytes + abi.SHARD_HANDLE_BYTES])
            caps = [int(np.ascontiguousarray(gathered[d, meta.nbytes + abi.SHARD_HANDLE_BYTES:]).view(np.uint64)[0]) for d in range(g)]
            _check_blob_sizes([self.e.blob_bytes(all_meta[s][d]) for s in range(g) for d in range(g)], "all-gathered")
            need = [sum(self.e.blob_bytes(all_meta[s][d]) for s in range(g)) for d in range(g)]
            if any(caps[d] < need[d] + 64 for d in range(g)):  # every rank sees the same numbers: all of them take this branch or none
                arena, handle, _ = self._guard(lambda: self.e.shard_arena(rnd, need[me]))
                h_out = torch.from_numpy(handle).to(self.device)
                h_all = torch.empty(g * abi.SHARD_HANDLE_BYTES, dtype=torch.uint8, device=self.device)
                dist.all_gather_into_tensor(h_all, h_out)  # also orders "arena (re)allocated" before anybody's stores
                handles = h_all.cpu().numpy().reshape(g, abi.SHARD_HANDLE_BYTES)
            self._guard(lambda: self.e.shard_open_peers(rnd, handles))
            return all_meta, arena
        all_meta, arena = self._timed(f"meta{rnd}", gather)
        # gar_shard_pack_peers returns after its streams have drained: this rank's blobs are in the peers' arenas.  _guard's
        # all-reduce (or the barrier) then makes "every rank has packed" known to every rank
        def pack():
            self._guard(lambda: self.e.shard_pack_peers(rnd, all_meta))
            if not self.check_errors:
                dist.barrier()
        self._timed(f"pack{rnd}", pack)
        self.bytes_sent += int(sum(int(x) for k, x in enumerate(nbytes) if k != me))
        self._timed(f"unpack{rnd}", lambda: self._guard(lambda: self.e.shard_unpack(rnd, arena, np.ascontiguousarray(all_meta[:, me]))))
