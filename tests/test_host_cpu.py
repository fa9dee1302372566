"""CPU-side tests (no GPU): the C-ABI library loads and exports every declared symbol, fails loudly without a
device, and the product's host logic (route codec, validators, workload generator, result re-hydration) agrees
with the oracle byte for byte."""
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    import bifromq_b200
    if not os.path.exists(os.path.join(ROOT, "bifromq_b200", "libbfq_gpumatch.so")):
        g.build()
    bifromq_b200.load_library()
    return bifromq_b200


def test_library_exports_every_declared_symbol(pkg):
    header = open(os.path.join(ROOT, "include", "bfq_gpumatch.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(bfq_[a-z_0-9]+)\s*\(", header))
    assert len(declared) >= 40
    from bifromq_b200 import _native
    raw = C.CDLL(_native.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(raw, s)]
    assert missing == []
    # and the Python binding covers the whole header
    assert declared == set(_native._SIGNATURES)


def test_no_cpu_fallback_without_device(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(pkg.NativeError) as ei:
        pkg.GpuRouteIndex(0)
    assert "no CPU fallback" in str(ei.value) or "CUDA" in str(ei.value)


def test_product_package_does_not_touch_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "bifromq_b200")):
        if "_build" in dirpath:
            continue
        for f in files:
            if f.endswith((".py", ".cc", ".cu", ".h", ".cuh")) or f == "Makefile":
                src = open(os.path.join(dirpath, f), errors="replace").read()
                for needle in ("oracle/", "oracle_lib", "liboracle", "import oracle", "from oracle", "oracle.h", "orc_"):
                    assert needle not in src, "%s must not use the oracle (%s)" % (f, needle)
    # neither do the helper scripts; only tests/, __graft_entry__.smoke() and bench.py's CPU legs may
    for f in os.listdir(os.path.join(ROOT, "tools")):
        src = open(os.path.join(ROOT, "tools", f), errors="replace").read()
        for needle in ("oracle_lib", "liboracle", "import oracle", "from oracle"):
            assert needle not in src, "tools/%s must not use the oracle (%s)" % (f, needle)
    bench = open(os.path.join(ROOT, "bench.py")).read()
    uses = [i for i in range(len(bench)) if bench.startswith("import oracle_lib", i)]
    assert uses, "bench.py times the oracle for cpu_baseline / --impl reference"
    for i in uses:   # the one place: oracle_for_sample(), called by run_cpu_baseline() only (cpu_baseline and --impl reference)
        head = bench[:i]
        fn = head[head.rindex("\ndef ") + 5:].split("(")[0]
        # forward configs / the inverse config C5: both are cpu_baseline / --impl reference legs, nothing the GPU arm calls
        assert fn in ("oracle_for_sample", "inverse_cpu_baseline"), "bench.py imports the oracle in %s()" % fn


# ------------------------------------------------------------------ codec parity (product C++ vs oracle C++)
def _rand_str(rng, alphabet, lo, hi):
    return "".join(rng.choice(alphabet) for _ in range(rng.randint(lo, hi)))


def test_route_key_codec_matches_oracle(pkg):
    from bifromq_b200 import schema
    rng = random.Random(3)
    alpha = "abcXYZ019_-$ .你好é😄"
    for _ in range(400):
        tenant = _rand_str(rng, "tenantABC01", 1, 12)
        levels = []
        for i in range(rng.randint(1, 6)):
            r = rng.random()
            levels.append("+" if r < 0.2 else ("" if r < 0.3 else _rand_str(rng, alpha, 1, 8)))
        if rng.random() < 0.2:
            levels.append("#")
        tf = "/".join(levels)
        url = schema.receiver_url(rng.choice([0, 1, 2, -7, 12345]), _rand_str(rng, alpha, 1, 20), _rand_str(rng, alpha, 0, 9))
        assert url == O.receiver_url(int(url.split(b"\0")[0]), url.split(b"\0")[1], url.split(b"\0")[2])
        assert schema.route_key(tenant, tf, url) == O.route_key(tenant, tf, url)
        for pre in ("$share/", "$oshare/"):
            g = _rand_str(rng, "groupAB12你", 1, 8)
            assert schema.route_key(tenant, pre + g + "/" + tf) == O.route_key(tenant, pre + g + "/" + tf)
        assert schema.tenant_begin_key(tenant) == O.tenant_begin_key(tenant)


def test_worked_key_example(pkg):  # SURVEY.md §8a
    from bifromq_b200 import schema
    url = schema.receiver_url(0, "inbox1", "d1")
    assert schema.route_key("t", "a/+", url) == bytes.fromhex("00000174" "6100" "2b00" "00" "c0" "01" "3000696e626f7831006431" "000b")
    assert schema.route_key("t", "$share/g1/a/#") == bytes.fromhex("00000174" "6100" "2300" "00" "aa" "02" "6731" "0002")


def test_validators_match_oracle(pkg):
    from bifromq_b200 import schema
    import test_oracle_golden as G  # reuse the TopicUtilsTest vectors by running the same inputs through both
    rng = random.Random(5)
    alpha = "ab/+#$\0 你😄/"
    cases = [("/", 40, 16, 255), ("", 40, 16, 255), ("$share/a/", 5, 4, 10), ("$share/g//+/a/#", 10, 4, 100),
             ("/a+/", 40, 16, 255), ("$oshare/g/#", 10, 4, 100), ("abc", 4, 1, 255), ("/abcde/fghij", 5, 4, 10)]
    for _ in range(3000):
        s = _rand_str(rng, alpha, 0, 14)
        if rng.random() < 0.2:
            s = rng.choice(["$share/", "$oshare/", "$share", "$shared/"]) + s
        cases.append((s, rng.randint(1, 6), rng.randint(1, 5), rng.randint(1, 20)))
    for s, a, b, c in cases:
        assert schema.is_valid_topic(s, a, b, c) == O.is_valid_topic(s, a, b, c), repr(s)
        assert schema.is_valid_topic_filter(s, a, b, c) == O.is_valid_topic_filter(s, a, b, c), repr(s)
    assert G.LOCAL_FIXTURES  # imported module is the golden-vector file


def test_python_rehydration_matches_oracle(pkg):
    from bifromq_b200 import schema
    rng = random.Random(8)
    for _ in range(100):
        tf = "/".join(rng.choice(["a", "+", "", "你好", "b1"]) for _ in range(rng.randint(1, 4)))
        url = O.receiver_url(rng.choice([0, 1, 5]), "rcv%d" % rng.randint(0, 99), "dk")
        k, v = O.route_key("tenantZ", tf, url), O.incarnation_bytes(rng.randint(0, 2 ** 40))
        m, o = schema.build_match_route(k, v), O.build_match_route(k, v)
        assert (m.tenant_id, m.mqtt_topic_filter, m.receiver_url, m.incarnation) == \
               (o["tenantId"], o["mqttTopicFilter"], o["receiverUrl"], o["incarnation"])
        assert schema.sub_broker_id(m) == o["subBrokerId"]
        members = {O.receiver_url(1, "m%d" % i, "d"): rng.randint(0, 2 ** 33) for i in range(rng.randint(0, 4))}
        full = rng.choice(["$share/", "$oshare/"]) + "grp/" + tf
        k, v = O.route_key("tenantZ", full), O.route_group(members)
        assert v == schema.route_group_bytes(members)
        m, o = schema.build_match_route(k, v), O.build_match_route(k, v)
        assert (m.tenant_id, m.mqtt_topic_filter, dict(m.members)) == (o["tenantId"], o["mqttTopicFilter"], o["members"])
        assert m.ordered == full.startswith("$oshare/")


# ------------------------------------------------------------------ workload generator
@pytest.mark.parametrize("config,scale", [("C1", 1.0), ("C2", 0.01), ("C3", 0.003), ("C4", 0.003)])
def test_workload_is_deterministic_sorted_and_decodable(pkg, config, scale):
    from bifromq_b200.workload import Workload
    w1, w2 = Workload(config, scale=scale), Workload(config, scale=scale, nthreads=1)
    assert w1.n_routes == w2.n_routes and w1.n_topics == w2.n_topics
    assert np.array_equal(w1.keys[:w1.key_off[-1]], w2.keys[:w2.key_off[-1]])
    assert np.array_equal(w1.topics[:w1.topic_off[-1]], w2.topics[:w2.topic_off[-1]])
    kb = w1.keys.tobytes()
    keys = [kb[w1.key_off[i]:w1.key_off[i + 1]] for i in range(w1.n_routes)]
    assert all(a < b for a, b in zip(keys, keys[1:])), "KV must be strictly ascending in byte order"
    vb = w1.vals.tobytes()
    tenants = set(w1.tenants)
    for i in range(0, w1.n_routes, max(1, w1.n_routes // 200)):
        m = O.build_match_route(keys[i], vb[w1.val_off[i]:w1.val_off[i + 1]])
        assert m["tenantId"] in tenants
        assert O.is_valid_topic_filter(m["mqttTopicFilter"], 40, 16, 255)
    for t in w1.topic_list()[:200]:
        assert O.is_valid_topic(t, 40, 16, 255)
    # most publish topics hit at least one filter (80% are derived from a filter)
    kv = O.KV()
    kv.load(w1.keys, w1.key_off, w1.vals, w1.val_off)
    tb, toff = O.blob(w1.tenants)
    out = kv.match_blobs(tb, toff, w1.topics, w1.topic_off, np.ascontiguousarray(w1.topic_tenant), w1.n_topics,
                         2 ** 31 - 1, 100, O.MODE_TRIE, False, 4)
    assert float((np.diff(out.offsets) > 0).mean()) > 0.6


def test_workload_sharding_partitions_the_tenants(pkg):
    from bifromq_b200.workload import Workload
    full = Workload("C3", scale=0.003)
    shards = [Workload("C3", scale=0.003, shard_index=i, shard_count=3) for i in range(3)]
    assert sorted(t for s in shards for t in s.tenants) == sorted(full.tenants)
    assert sum(s.n_routes for s in shards) == full.n_routes
    assert sum(s.n_topics for s in shards) == full.n_topics


def test_workload_c5_shapes(pkg):
    from bifromq_b200.workload import Workload
    w = Workload("C5", scale=0.005)
    assert w.n_routes == 0 and w.n_topics > 0 and w.n_query_filters > 0
    fs = w.query_filter_list()
    assert all((b"+" in f) or f.endswith(b"/#") for f in fs)
    assert all(O.is_valid_topic_filter(f, 40, 16, 255) for f in fs[:300])


def test_bench_roofline_record_and_defaults():
    """bench.py's pure-host pieces: the roofline record follows SURVEY.md §8(d) and the default run is the full-size C4 line"""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    ns, n = 1000, 1_000_000
    st = {"V": 25.0 * ns, "P": 70.0 * ns, "ranges": 6.0 * ns, "R": 300.0 * ns}
    r = bench.make_roofline(50 * ns, st, ns, n, 0.5)
    per_topic = 50 + 4 + 32 * 25.0 + 8 * 70.0 + 8 * 6.0 + 4
    assert abs(r["alg_bytes_per_topic"] - per_topic) < 1e-9
    assert abs(r["achieved"] - per_topic * n / 0.5e-3 / 1e9) < 1e-6
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(r["frac_of_nominal_8000"] - r["achieved"] / 8000.0) < 1e-12
    traffic = json.load(open(os.path.join(ROOT, "profiles", "latest_kernel_traffic.json")))["dram_bytes_per_launch"]
    assert r["traffic"] == traffic and abs(r["dram_gbs_from_ncu_traffic"] - traffic / 0.5e-3 / 1e9) < 1e-6
    assert bench.METRIC.startswith("publish-topics matched/sec")
    assert bench._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert bench.pin_to_gpu_numa_node(0) is None      # no GPU here: must decline quietly, never raise


def test_bench_dump_outputs_sample(tmp_path):
    """bench.py --dump-outputs: the rows of the seeded sample are the same every run, each row's values come out sorted (the
    device CSR leaves them unordered), the values are cut at the budget and the files are float64 .npy; an empty output (no
    throttle event, say) is left out rather than written empty"""
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(1)
    off = np.zeros(1001, np.int64)
    off[1:] = np.cumsum(rng.integers(0, 9, 1000))
    vals = rng.integers(0, 2 ** 32, int(off[-1]), dtype=np.int64)
    pick = bench.cpu_sample_indices(1000, 100)
    assert np.array_equal(pick, bench.cpu_sample_indices(1000, 100)) and len(np.unique(pick)) == 100
    assert np.array_equal(bench.cpu_sample_indices(50, 100), np.arange(50))
    got_off, got = bench.sample_csr(torch.from_numpy(off), torch.from_numpy(vals), torch.from_numpy(pick), 250)
    rows = [sorted(vals[off[i]:off[i + 1]].tolist()) for i in pick]
    assert got_off.tolist() == [0] + np.cumsum([len(r) for r in rows]).tolist()
    flat = [v for r in rows for v in r]
    assert len(flat) > 250 and got.tolist() == flat[:250]
    bench.write_dump(str(tmp_path / "out"), {"offsets": got_off, "ranks": got, "topics": pick, "throttled": np.zeros((0, 3), np.int32)})
    ranks = np.load(str(tmp_path / "out" / "ranks.npy"))
    assert ranks.dtype == np.float64 and ranks.tolist() == flat[:250]
    assert sorted(os.listdir(str(tmp_path / "out"))) == ["offsets.npy", "ranks.npy", "topics.npy"]


def _route_blobs(pairs):
    keys = b"".join(k for k, _ in pairs)
    vals = b"".join(v for _, v in pairs)
    koff = np.zeros(len(pairs) + 1, np.int64)
    voff = np.zeros(len(pairs) + 1, np.int64)
    koff[1:] = np.cumsum([len(k) for k, _ in pairs])
    voff[1:] = np.cumsum([len(v) for _, v in pairs])
    return (np.frombuffer(keys, np.uint8).copy(), koff, np.frombuffer(vals or b"\0", np.uint8).copy(), voff)


def test_builder_places_every_child_array_kind():
    """host builder + its self-check (every placed node is found again from its parent's record the way the kernels look it
    up) over fan-outs of 1, 3, 16, 17, 40, 300 (perfect-hashed private arrays) and 1500 / 2500 (global tag table)"""
    from bifromq_b200 import _native as N, schema
    pairs = []
    widths = {"w1": 1, "w3": 3, "w16": 16, "w17": 17, "w40": 40, "w300": 300, "w1500": 1500}
    for name, n in widths.items():
        for i in range(n):
            url = schema.receiver_url(i % 2, "r%s%d" % (name, i), "d")
            pairs.append((schema.route_key("t", "%s/c%04d" % (name, i), url), schema.incarnation_bytes(1)))
        pairs.append((schema.route_key("t", "%s/+" % name, schema.receiver_url(0, "p" + name, "d")), schema.incarnation_bytes(1)))
    for i in range(2500):
        pairs.append((schema.route_key("t2", "dev%05d/state" % i, schema.receiver_url(0, "s%d" % i, "d")), schema.incarnation_bytes(1)))
    pairs.sort()
    k, ko, v, vo = _route_blobs(pairs)
    st = np.zeros(16, np.int64)
    rc = N.lib.bfq_host_build_stats(k.ctypes.data, ko.ctypes.data, v.ctypes.data, vo.ctypes.data, len(pairs), st.ctypes.data, 16)
    assert rc == 0, N.lib.bfq_last_error()
    assert st[0] == len(pairs) and st[1] == 2
    n_nodes = int(st[2])
    # 2 roots + per width: the width node, its children, its '+' child; t2: 2500 devices each with a "state" child
    assert n_nodes == 2 + sum(1 + n + 1 for n in widths.values()) + 2 * 2500
    assert st[3] >= n_nodes - 2            # slots: private arrays + tag-table blocks
    assert st[9] + st[10] + st[11] + st[12] + st[13] == n_nodes   # child-count histogram covers every node


def test_jni_shim_covers_every_native_method_and_type_checks():
    """jni/bfq_gpumatch_jni.c (the shim a maintainer adds) defines one function per `static native` method of
    jni/java/.../BfqNative.java, calls only functions include/bfq_gpumatch.h declares, and compiles against the JNI stand-in
    header (no JDK in this image; __graft_entry__.build() runs the same check)"""
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    java = open(os.path.join(root, "jni", "java", "org", "apache", "bifromq", "dist", "worker", "gpumatch", "BfqNative.java")).read()
    csrc = open(os.path.join(root, "jni", "bfq_gpumatch_jni.c")).read()
    natives = set(re.findall(r"static native [\w\[\]]+ (\w+)\(", java))
    defined = set(re.findall(r"JFN\((\w+)\)\(", csrc))
    assert natives and natives == defined, (natives - defined, defined - natives)
    header = open(os.path.join(root, "include", "bfq_gpumatch.h")).read()
    declared = set(re.findall(r"\b(bfq_\w+)\s*\(", header))
    called = set(re.findall(r"\b(bfq_\w+)\s*\(", csrc)) - {"bfq_gpumatch_jni"}
    assert called <= declared, called - declared
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-DBFQ_JNI_STUB",
                           os.path.join(root, "jni", "bfq_gpumatch_jni.c")])


def test_retain_key_codec_matches_the_oracle():
    """bfq_retain_key / bfq_retain_key_prefix (csrc/codec.cc) against the oracle's restatement of the retain store schema, on
    random topics and filters incl. empty levels and non-ASCII text (UTF-16 code units drive LevelHash)"""
    import random
    from bifromq_b200 import schema
    rng = random.Random(3)
    vocab = ["a", "b", "", "dd", "é", "温度", "x" * 30, "$sys", "😀"]
    for _ in range(1500):
        tenant = rng.choice(["t", "tenantA", "租户"])
        lv = [rng.choice(vocab) for _ in range(rng.randint(1, 7))]
        topic = "/".join(lv)
        assert schema.retain_key(tenant, topic) == O.retain_key(tenant, topic), topic
        f = list(lv)
        for i in range(len(f)):
            if rng.random() < 0.25:
                f[i] = "+"
        if rng.random() < 0.3:
            f[-1] = "#"
        tf = "/".join(f)
        assert schema.retain_key_prefix(tenant, tf) == O.retain_key_prefix(tenant, tf), tf


_BUILDER_AB_CHILD = r"""
import sys, json, random
import numpy as np
sys.path.insert(0, %(root)r)
from bifromq_b200 import _native as N, schema
rng = random.Random(20260923)
LONG = "L" * 24                                    # levels longer than one 24-byte token share chunk nodes
names = ["", "a", "b", "ab", "a\x01", "\x01", "\x02x", "+", "zz", LONG + "p", LONG + "q", LONG + LONG + "r", LONG]
pairs = {}
for tenant in ("t", "t0", "u"):
    for _ in range(1500):
        depth = rng.randint(1, 5)
        levels = [rng.choice(names) for _ in range(depth)]
        if rng.random() < 0.25:
            levels.append("#")
        tf = "/".join(levels)
        if tf.startswith("$") or tf == "":
            continue
        for _ in range(rng.randint(1, 4)):
            kind = rng.random()
            if kind < 0.15:
                key = schema.route_key(tenant, "$share/g%%d/%%s" %% (rng.randint(0, 3), tf), "")
                val = b"\x0a\x06\x0a\x02r1\x10\x01"
            else:
                # receiver urls starting with control bytes after the bucket byte: a parent's OWN keys then interleave with
                # the subtree of its empty-named child (the bucket-byte quirk), the revisit the sorted builder must survive
                url = schema.receiver_url(rng.randint(0, 1), "r%%d" %% rng.randint(0, 400), rng.choice(["d", "\x01d", "e"]))
                key = schema.route_key(tenant, tf, url)
                val = schema.incarnation_bytes(1)
            pairs[key] = val
pairs = sorted(pairs.items())
keys = b"".join(k for k, _ in pairs); vals = b"".join(v for _, v in pairs)
koff = np.zeros(len(pairs) + 1, np.int64); voff = np.zeros(len(pairs) + 1, np.int64)
koff[1:] = np.cumsum([len(k) for k, _ in pairs]); voff[1:] = np.cumsum([len(v) for _, v in pairs])
k = np.frombuffer(keys, np.uint8).copy(); v = np.frombuffer(vals, np.uint8).copy()
st = np.zeros(19, np.int64)
rc = N.lib.bfq_host_build_stats(k.ctypes.data, koff.ctypes.data, v.ctypes.data, voff.ctypes.data, len(pairs), st.ctypes.data, 19)
print(json.dumps({"rc": int(rc), "stats": st[:14].tolist(), "sum": int(st[16]), "same_as_concat": int(st[17]),
                  "tenant_images_equal": int(st[18]), "n": len(pairs)}))
"""


def test_sorted_order_trie_construction_builds_the_same_image_as_the_hash_table_one():
    """index_builder.cc builds a tenant's trie from the KV order alone (a child can only be its parent's most recent child) and
    keeps the hash-table construction as the checked fallback (BFQ_BUILDER=hash forces it). Both must produce the same image,
    byte for byte (stats[16] = checksum of records, tags, roots, segments and per-rank arrays) — on a key set with empty
    levels, control bytes, '+', '#', shared-subscription keys and long levels sharing 24-byte chunks, where a parent's own keys
    interleave with its empty-named child's subtree (the reference's bucket-byte quirk, DESIGN.md §2)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {}
    for mode in ("sorted", "hash", "pieces"):
        env = dict(os.environ)
        for k in ("BFQ_BUILDER", "BFQ_INSERT_PARALLEL_MIN", "BFQ_INSERT_THREADS"):
            env.pop(k, None)
        if mode == "hash":
            env["BFQ_BUILDER"] = "hash"
        if mode == "pieces":   # the several-thread insertion of large tenants, forced onto these small ones: cut at first-level
            env["BFQ_INSERT_PARALLEL_MIN"] = "2"   # boundaries (the empty first level, '+', control bytes among them), pieces
            env["BFQ_INSERT_THREADS"] = "5"        # concatenated
        r = subprocess.run([sys.executable, "-c", _BUILDER_AB_CHILD % {"root": root}], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        out[mode] = json.loads(r.stdout.strip().splitlines()[-1])
        assert out[mode]["rc"] == 0 and out[mode]["n"] > 5000
        # the full build straight from the staged per-tenant blobs (what bfq_index_commit runs) == the build from one
        # concatenated blob with a tenant-boundary scan
        assert out[mode]["same_as_concat"] == 1
        # the stand-alone image of every tenant (what a delta commit builds for a touched tenant, build_tenant_image) == its
        # part of the full image
        assert out[mode]["tenant_images_equal"] == out[mode]["stats"][1] == 3
    assert out["sorted"]["stats"] == out["hash"]["stats"] == out["pieces"]["stats"]
    assert out["sorted"]["sum"] == out["hash"]["sum"] == out["pieces"]["sum"] != 0
    assert out["sorted"]["stats"][6] > 0 and out["sorted"]["stats"][7] > 0   # multi-segment filters and long-token chunks occur


def test_staging_delta_merge_equals_a_sorted_map(tmp_path):
    """Staging::merge_tenant (the host half of bfq_index_apply + bfq_index_commit's delta path) copies the runs of base keys
    between two delta keys in bulk; tests/native/staging_merge_test.cc drives 200 rounds of random load / upsert / erase /
    merge over several tenants (new and vanishing ones included) against a std::map."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    csrc = os.path.join(root, "bifromq_b200", "csrc")
    exe = str(tmp_path / "staging_merge_test")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I" + csrc, os.path.join(root, "tests", "native", "staging_merge_test.cc"),
                           os.path.join(csrc, "index_builder.cc"), os.path.join(csrc, "codec.cc"), "-lpthread", "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "merge ok" in out.stdout, out.stdout + out.stderr
