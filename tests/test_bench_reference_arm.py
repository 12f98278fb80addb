"""The bench contract's reference arm (`bench.py --impl reference`) runs on the host cores only: its JSON line can be checked on
the CPU tier.  (The GPU arm of bench.py needs a B200 and is exercised by the driver / `gpurun`.)"""
import json
import subprocess
import sys
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent


def _run(*extra):
    out = subprocess.run([sys.executable, str(REPO / "bench.py"), "--impl", "reference", "--objects", "3000", "--steps", "2", "--warmup", "1", *extra],
                         capture_output=True, text=True, timeout=600, cwd=str(REPO))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run()
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "objects/s"
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1
    assert abs(d["ms_per_step"] * d["value"] / 1e3 - 3000) < 1e-3 * 3000  # value = objects / time of one step
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"]
    assert str(cb["cores"]) in cb["scaling"]                      # reported at a thread count of the ladder ...
    best = max(cb["scaling"].values())
    assert cb["scaling"][str(cb["cores"])] >= 0.5 * best          # ... the one the ladder pass found fastest (timing noise aside)
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["same_config"] is True and d["config"]["sample_objects"] == 3000
    assert cb["literal_port"]["value"] > 0


def test_byte_models_identify_keys_by_their_bytes(garecon):
    """bench.py's per-kernel byte models pick the system tags / the route53 annotation by comparing the key BYTES (a user tag of
    the same length must not be counted), and run on host tables alone."""
    import importlib
    import sys
    import numpy as np
    sys.path.insert(0, str(REPO))
    bench = importlib.import_module("bench")
    ANN = "aws-global-accelerator-controller.h3poteto.dev/"
    decoy_tag = "x" * 28                                     # as long as aws-global-accelerator-owner
    decoy_ann = "y" * 63                                     # as long as the route53-hostname annotation key
    objects = [dict(kind="service", ns="default", name=f"s{i}", spec_type="LoadBalancer", ports=[(80, "TCP")], lb_ingress=[f"{i:032x}-0123456789abcdef.elb.us-west-2.amazonaws.com"],
                    annotations={ANN + "route53-hostname": f"h{i}.example.com", decoy_ann: "z" * 500, ANN + "global-accelerator-managed": "true"}) for i in range(5)]
    accs = [{"arn": f"a{i}", "name": f"service-default-s{i}", "dns": f"a{i}.awsglobalaccelerator.com", "enabled": True,
             "tags": [("aws-global-accelerator-controller-managed", "true"), ("aws-global-accelerator-owner", f"service/default/s{i}"), (decoy_tag, "q" * 300),
                      ("aws-global-accelerator-target-hostname", "h" * 70), ("aws-global-accelerator-cluster", "default")],
             "listeners": []} for i in range(5)]
    snap = garecon.pack(objects, {"lbs": [], "accelerators": accs, "zones": []})
    o, a = snap.objects, snap.actual
    tk = bench._np_col(a.tag_key, a.n_tags, np.uint64)
    owner = bench._key_is(tk, a.slab, a.slab_len, bench.TAG_OWNER_KEY)
    assert owner.tolist() == [False, True, False, False, False] * 5             # the 28-byte decoy is not the owner tag
    ak = bench._np_col(o.ann_key, o.n_ann, np.uint64)
    assert int(bench._key_is(ak, o.slab, o.slab_len, bench.ANN_R53_KEY).sum()) == 5
    m = bench.kernel_byte_models(o, a, 5, 5, 1.0)
    assert all(isinstance(v, int) and v >= 0 for v in m.values()) and m["ga_objects"] > 0 and m["r53_pairs"] > 0
    big = bench.kernel_byte_models(o, a, 5, 5, 1.0)["digest_accelerators"]
    # the 300-byte decoy value is not part of what digest_accelerators must read: 5 x (4 + 18 + 70 + 7) system tag value bytes are
    sys_bytes = 5 * (len("true") + len("service/default/s0") + 70 + len("default"))
    assert big < sys_bytes + 5 * 300 + 16 * a.n_tags + 5 * 200


def test_dump_outputs_is_exact_and_sampled_the_same_way_every_time(garecon, oracle, tmp_path):
    """bench.py --dump-outputs: every change-set array as exact float64 (ops as rows of six fields, string references as offset and
    length); above the size cap a sample of rows that depends only on the row count."""
    import numpy as np
    import randmodel
    sys.path.insert(0, str(REPO))
    bench = __import__("bench")
    cs = oracle.diff(garecon.pack(*randmodel.make(3, n_objects=200)), "default", mode=1)
    assert len(cs.ops) > 40 and len(cs.tok_name) > 40
    rows = bench.dump_outputs(cs, tmp_path / "full")
    load = lambda d, k: np.load(tmp_path / d / f"{k}.npy")
    assert sorted(rows) == sorted(list(cs.ARRAYS) + ["counts"])
    for k in cs.ARRAYS:
        assert load("full", k).dtype == np.float64
    assert (load("full", "status_ga") == cs.status_ga).all() and (load("full", "dports") == cs.dports).all()
    assert (load("full", "ops").astype(np.uint32) == np.stack([cs.ops[f] for f in ("head", "obj", "sub", "a0", "a1", "a2")], axis=1)).all()
    name = load("full", "tok_name").astype(np.uint64)
    assert ((name[:, 1] << np.uint64(40)) | name[:, 0] == cs.tok_name).all()
    assert load("full", "counts").tolist() == [200, len(cs.ops), len(cs.tok_code), len(cs.dports)]
    for d in ("a", "b"):
        rows = bench.dump_outputs(cs, tmp_path / d, max_values=24)
    assert rows["status_ga"] == 24 and rows["ops"] == 4 and rows["tok_name"] == 12 and rows["section_begin"] == 5
    for k in rows:
        assert np.array_equal(load("a", k), load("b", k))
    full_ops, ops = load("full", "ops"), load("a", "ops")
    at = [next(i for i in range(len(full_ops)) if (full_ops[i] == r).all()) for r in ops]
    assert at == sorted(at)


def test_bench_rejects_zero_steps_and_dumps_it_cannot_make():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"], ["--mode", "sharded", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, str(REPO / "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=str(REPO))
        assert out.returncode == 2 and "error" in out.stderr, extra
