"""CPU-side checks of libcitus_gpu.so: the library loads, exports every symbol the header
declares, and its host logic (shard writer, chunk-group skipping, bounds, numeric text)
agrees with the oracle / the reference goldens.  No kernel is launched here."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cg():
    from citus_b200 import build
    build.build()
    from citus_b200 import capi, columnar
    capi.lib()
    return columnar


def test_library_exports_every_declared_symbol(cg):
    from citus_b200 import capi
    header = open(os.path.join(ROOT, "include", "citus_gpu.h")).read()
    declared = set(re.findall(r"\b(cg_[a-z0-9_]+)\s*\(", header))
    declared.discard("cg_partial_dense_touch")     # mentioned in a comment only
    L = C.CDLL(capi.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, missing
    bound = {name for name, _, _ in capi.SYMBOLS}
    assert declared <= bound, declared - bound


def test_no_oracle_in_product():
    # the product tree must never import, link or execute anything under oracle/
    for base, _, files in os.walk(os.path.join(ROOT, "citus_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".cuh")):
                text = open(os.path.join(base, f), errors="ignore").read()
                assert "liboracle" not in text and "import oracle" not in text and "from oracle" not in text, f


def test_calls_fail_loudly_without_init(cg):
    # in a process of its own: the GPU tests of the same session may already have called cg_init in this one
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, sys.argv[1])\n"
            "from citus_b200 import capi, columnar as cg\n"
            "try:\n"
            "    cg.GpuColumnarAgg(cg.make_desc(aggs=[cg.count_star()]), [(8, 0)])\n"
            "except capi.CitusGpuError as e:\n"
            "    print('refused:', e)\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("refused:") and "cg_init" in r.stdout, r.stdout + r.stderr


def _same_image(rel, t):
    """product writer image == oracle writer image (payloads, pd_lower, stripes, skip nodes)"""
    a = rel.pages().reshape(-1, 8192)
    b = t.pages().reshape(-1, 8192)
    assert a.shape == b.shape
    assert np.array_equal(a[2:, 24:], b[2:, 24:])
    assert np.array_equal(a[2:, 12:14], b[2:, 12:14])          # pd_lower
    assert np.array_equal(rel.stripes_bytes(), t.stripes_array())
    assert np.array_equal(rel.nodes_bytes(), t.nodes_array())


def test_writer_matches_oracle_writer_byte_for_byte(cg, oracle):
    rng = np.random.default_rng(11)
    n = 23456
    a = rng.integers(-2**40, 2**40, n)
    b = rng.integers(-100, 100, n)
    c = rng.integers(0, 2, n)
    d = rng.integers(-2**31, 2**31, n)
    nb = (rng.random(n) < 0.2).astype(np.uint8)
    nd = (rng.random(n) < 0.9).astype(np.uint8)
    nd[5000:7000] = 1                                          # whole chunks all-NULL: no min/max
    rel = cg.Relation.write([8, 4, 2, 1], [a, b, c, d % 100], [None, nb, None, nd],
                            stripe_row_limit=5000, chunk_row_limit=1000)
    t = oracle.Table([8, 4, 2, 1], stripe_row_limit=5000, chunk_row_limit=1000)
    t.insert([a, b, c, d % 100], nulls=[None, nb, None, nd])
    _same_image(rel, t)
    # the oracle's row-at-a-time reader decodes the product image back to the inputs
    t2 = oracle.Table.attach(rel.pages(), rel.stripes_bytes(), rel.nodes_bytes(), [8, 4, 2, 1], chunk_row_limit=1000)
    vals, nulls = t2.decode_all()
    assert np.array_equal(vals[0], a) and np.array_equal(vals[2], c)
    assert np.array_equal(nulls[1], nb) and np.array_equal(vals[1][nb == 0], b[nb == 0])
    assert np.array_equal(nulls[3], nd)
    # columnar.compression = lz4: both writers hand every value stream to the same LZ4_compress_default
    if oracle.lib().orc_have_lz4():
        cg.set_writer_compression("lz4")
        try:
            rel = cg.Relation.write([8, 4, 2, 1], [a, b, c, d % 100], [None, nb, None, nd],
                                    stripe_row_limit=5000, chunk_row_limit=1000)
        finally:
            cg.set_writer_compression("none")
        t = oracle.Table([8, 4, 2, 1], stripe_row_limit=5000, chunk_row_limit=1000, compression=oracle.COMP_LZ4)
        t.insert([a, b, c, d % 100], nulls=[None, nb, None, nd])
        assert any(nd_.compression_type == oracle.COMP_LZ4 for nd_ in t.nodes())
        _same_image(rel, t)
    if oracle.lib().orc_have_zstd():
        cg.set_writer_compression("zstd")
        try:
            rel = cg.Relation.write([8, 4, 2, 1], [a, b, c, d % 100], [None, nb, None, nd],
                                    stripe_row_limit=5000, chunk_row_limit=1000)
        finally:
            cg.set_writer_compression("none")
        t = oracle.Table([8, 4, 2, 1], stripe_row_limit=5000, chunk_row_limit=1000, compression=oracle.COMP_ZSTD)
        t.insert([a, b, c, d % 100], nulls=[None, nb, None, nd])
        assert any(nd_.compression_type == oracle.COMP_ZSTD for nd_ in t.nodes())
        _same_image(rel, t)


def test_float_columns_and_default_limits(cg, oracle):
    rng = np.random.default_rng(5)
    n = 310001                                                 # 3 stripes, last chunk of 1 row
    f8 = rng.normal(size=n)
    f4 = rng.normal(size=n).astype(np.float32).astype(np.float64)
    i8 = np.arange(n)
    rel = cg.Relation.write([8, 4, 8], [f8, f4, i8], type_classes=[1, 1, 0])
    t = oracle.Table([8, 4, 8], atttype=[1, 1, 0])
    t.insert([f8, f4, i8])
    _same_image(rel, t)
    assert rel.view.nstripes == 3 and rel.view.stripes[2].chunk_count == 2


def test_generated_relation_is_reproducible_and_decodable(cg, oracle):
    cols = [(8, 0, 0, 1000, 0), (8, 0, -10**9, 10**9, 50000), (4, 1, 7, 0, 0), (2, 0, -5, 5, 0)]
    rel = cg.Relation.generate(cols, 45678, seed=20260922, first_row=1000, stripe_row_limit=20000,
                               chunk_row_limit=5000, nthreads=4)
    rel2 = cg.Relation.generate(cols, 45678, seed=20260922, first_row=1000, stripe_row_limit=20000,
                                chunk_row_limit=5000, nthreads=1)
    assert np.array_equal(rel.pages(), rel2.pages())
    t = oracle.Table.attach(rel.pages(), rel.stripes_bytes(), rel.nodes_bytes(), [8, 8, 4, 2], chunk_row_limit=5000)
    vals, nulls = t.decode_all()
    sm = oracle.lib().orc_splitmix64
    # the generator is the published splitmix64 counter scheme (include/citus_gpu.h)
    for row in (0, 1, 777, 45677):
        h = sm(20260922 ^ (0 << 56) ^ (1000 + row))
        assert vals[0][row] == h % 1000
        h1 = sm(20260922 ^ (1 << 56) ^ (1000 + row))
        isnull = sm((~20260922 & (2**64 - 1)) ^ (1 << 56) ^ (1000 + row)) % 1000000 < 50000
        assert bool(nulls[1][row]) == isnull
        if not isnull:
            assert vals[1][row] == -10**9 + h1 % (2 * 10**9)
        assert vals[2][row] == 7 + 1000 + row
    assert 0.03 < nulls[1].mean() < 0.07
    assert vals[0].min() >= 0 and vals[0].max() < 1000
    # re-encoding the decoded rows with the oracle's writer reproduces the image
    t2 = oracle.Table([8, 8, 4, 2], stripe_row_limit=20000, chunk_row_limit=5000)
    t2.insert(vals, nulls=nulls)
    _same_image(rel, t2)


def _mask_count(cg, rel, quals, pushdown=True):
    from citus_b200.capi import lib, check
    d = cg.make_desc(quals=quals, aggs=[cg.count_star()], qual_pushdown=pushdown)
    total = 0
    for s in range(rel.view.nstripes):
        mask = np.zeros(rel.view.stripes[s].chunk_count, np.uint8)
        f = C.c_int64()
        check(lib().cg_selected_chunk_mask(C.byref(rel.view), s, C.byref(d), mask.ctypes.data, C.byref(f)))
        assert f.value == int((mask == 0).sum())
        total += f.value
    return total


def test_selected_chunk_mask_goldens(cg, expected, oracle):
    for case in expected["simple_chunk_filtering"]:
        rel = cg.Relation.write([4], [np.arange(0, case["max"] + 1)])
        assert _mask_count(cg, rel, [(0, ">", case["gt"])]) == case["groups_removed"]
        assert _mask_count(cg, rel, [(0, ">", case["gt"])], pushdown=False) == 0
    case = expected["multi_column_chunk_filtering"]
    i = np.arange(0, case["max"] + 1)
    rel = cg.Relation.write([4, 4], [i, i + 1])
    assert _mask_count(cg, rel, [(0, ">", 50000)]) == case["groups_removed"]
    assert _mask_count(cg, rel, [(0, ">", 50000), (1, ">", 50000)]) == case["groups_removed"]
    rel = cg.Relation.write([4, 4], [np.arange(6), np.zeros(6)], [None, np.ones(6, np.uint8)])
    assert _mask_count(cg, rel, [(0, ">", 50000), (1, ">", 50000)]) == 1
    assert _mask_count(cg, rel, [(1, ">", 50000)]) == 0       # all-NULL chunk has no min/max
    # differential: every operator against the oracle on random data
    rng = np.random.default_rng(2)
    a = np.sort(rng.integers(0, 10000, 30000))
    b = rng.integers(0, 100, 30000)
    rel = cg.Relation.write([8, 8], [a, b], stripe_row_limit=7000, chunk_row_limit=1000)
    t = oracle.Table.attach(rel.pages(), rel.stripes_bytes(), rel.nodes_bytes(), [8, 8], chunk_row_limit=1000)
    for op in ("<", "<=", "=", ">=", ">", "<>"):
        for k in (-1, 0, 2500, 5000, 9999, 10000):
            quals = [(0, op, k), (1, "<", 50)]
            assert _mask_count(cg, rel, quals) == t.scan(quals, aggs=[oracle.count_star()]).chunk_groups_filtered


def test_relation_bounds(cg):
    n = 25000
    key = np.arange(n) % 777 + 5
    v = np.arange(n) - 12000
    rel = cg.Relation.write([8, 8], [key, v], stripe_row_limit=10000, chunk_row_limit=1000)
    d = cg.make_desc(quals=[(1, "<", 0)], group_cols=[0], aggs=[cg.count_star(), cg.sum_(1)])
    kmin, kmax, bounds, rows = cg.relation_bounds(rel, d)
    assert (kmin, kmax) == (5, 781)
    assert rows == 12000                       # chunk groups with v >= 0 are skipped
    assert bounds[1] == 12000 and bounds[0] == 0


def test_numeric_text_goldens(cg, expected, oracle):
    assert cg.numeric_out(2432777858, 4) == expected["tpch_q6"]
    assert cg.numeric_out(-5, 2) == "-0.05" and cg.numeric_out(0, 2) == "0.00" and cg.numeric_out(-(2**100), 0) == str(-(2**100))
    assert cg.numeric_div_out(18755, 0, 8) == expected["contestant_avg"]
    # Q1's avg columns: sum (scale 2) / count
    q1 = expected["tpch_q1"]
    def cents(s):
        return int(s.replace(".", ""))
    for row in q1:
        n = int(row[9])
        assert cg.numeric_div_out(cents(row[2]), 2, n) == row[6]
        assert cg.numeric_div_out(cents(row[3]), 2, n) == row[7]
    # differential against the oracle's decimal implementation
    rng = np.random.default_rng(9)
    for _ in range(300):
        v = int(rng.integers(-10**17, 10**17)) * int(rng.integers(1, 10**6))
        s = int(rng.integers(0, 7))
        c = int(rng.integers(1, 10**9))
        assert cg.numeric_div_out(v, s, c) == oracle.numeric_div_str(v, s, c, 0), (v, s, c)
        assert cg.numeric_out(v, s) == oracle.numeric_str(v, s)


# --------------------------------------------------------------------------- plan-specialised kernels (NVRTC)
def _jit_check(cg, quals, group, aggs, lens, kmin, kmax, rows, float_cols=()):
    from citus_b200 import capi
    d = cg.make_desc(quals, group, aggs, float_cols=float_cols)
    cols = (capi.CgColumnDesc * len(lens))()
    for i, l in enumerate(lens):
        cols[i].attlen, cols[i].type_class = l, (1 if i in float_cols else 0)
    kind = C.c_int32(-1)
    buf = C.create_string_buffer(1 << 18)
    rc = capi.lib().cg_jit_compile_check(C.byref(d), cols, len(lens), kmin, kmax, rows, C.byref(kind), buf, len(buf))
    assert rc == 0, capi.lib().cg_last_error().decode()
    return kind.value, buf.value.decode()


def test_jit_generates_valid_sm100a_code_for_every_plan_form(cg):
    """cg_jit.cpp: the CUDA generated for a query shape compiles (NVRTC cross-compiles without a GPU);
    the struct text inside it must match the host's KPlan (static_assert on the sizes)"""
    try:
        C.CDLL("libnvrtc.so.12")
    except OSError:
        pytest.skip("libnvrtc missing")
    # C2 shape: direct-indexed table in global memory
    kind, src = _jit_check(cg, [(1, "<", 50)], [0], [cg.sum_(2), cg.count_star()], [8] * 8, 0, 999_999, 10**9)
    assert kind == 2 and "red_add(e" in src and "cg_jit_scan" in src
    # hash table, min/max, <> qual
    kind, src = _jit_check(cg, [(1, "<", 50), (3, "<>", 7)], [0], [cg.sum_(2), cg.count_star(), cg.min_(2), cg.max_(3)],
                           [8] * 8, 0, -1, 10**9)
    assert kind == 2 and "hash_slot_slow(P, key, h)" in src and "atomicMin" in src
    # plain aggregate over mixed widths: thread registers + warp shuffles
    kind, src = _jit_check(cg, [(1, "<", 50)], [], [cg.sum_(2), cg.count_star(), cg.count(3), cg.min_(4), cg.max_(5)],
                           [8, 4, 2, 1, 8, 8], 0, -1, 10**9)
    assert kind == 0 and "__shfl_xor_sync" in src
    # TPC-H Q1 shape: 6 slots x (rows + 5 bounded sums) -> one shared-memory cell per lane and word
    q1 = [cg.sum_(0), cg.sum_(1), cg.Agg(2, [(1, 0, 1), (2, 100, -1)]), cg.Agg(2, [(1, 0, 1), (2, 100, -1), (3, 100, 1)]),
          cg.sum_(2), cg.count_star()]
    for a, b in zip(q1, (5100, 10_500_000, 10**9, 2 * 10**11, 11, 0)):
        a.term_abs_bound = b
    kind, src = _jit_check(cg, [(6, "<=", -486)], [4, 5], q1, [8, 8, 8, 8, 1, 1, 4, 4], 65 | (70 << 32), 67 | (71 << 32), 6 * 10**8)
    assert kind == 1 and "s_acc" in src and "P.aggs[3].b[2]" in src
    # float4 / float8 columns: btree comparison with NaN ordering, ordered min/max
    kind, src = _jit_check(cg, [(1, ">=", 0)], [0], [cg.sum_(1, True), cg.min_(1, True), cg.max_(2, True), cg.count_star()],
                           [4, 8, 4], 0, 10**6, 10**6, float_cols=(1, 2))
    assert "fcmp(v" in src and "f8_ordered" in src and "__uint_as_float" in src


def test_run_time_options_are_named(cg):
    """cg_set_option: every documented switch is accepted, anything else is an error (no silent typos)"""
    from citus_b200 import capi
    for name, value in (("jit", 1), ("force_general", 0), ("realign_tma", 1), ("peer_window", 1), ("lz4_lanes", -1), ("lz4_lane_warps", 64)):
        cg.set_option(name, value)
    with pytest.raises(capi.CitusGpuError) as e:
        cg.set_option("lz4_lane", 1)
    assert e.value.code == capi.CG_EINVAL
    assert capi.lib().cg_comm_peer_window() == 0          # no communicator in this process


# --------------------------------------------------------------------------- repartition exchange, peer-window layout
@pytest.mark.parametrize("P,W", [(32, 8), (32, 2), (7, 4), (3, 8), (1, 1), (33, 16), (32, 5)])
def test_peer_plan_fills_every_receive_buffer_in_order(P, W):
    """cg_comm_peer_plan (pure host arithmetic): all W ranks of a repartition modelled in one process.  Every rank
    "stores" its rows where the plan says; every receive buffer must come out exactly filled, in (source rank, local
    partition) order, which is the layout of the ncclSend/ncclRecv form and what cg_comm_exchange_result describes"""
    from citus_b200 import distributed as cgd
    rng = np.random.default_rng(P * 100 + W)
    counts = rng.integers(0, 50, size=(W, P)) * (rng.random((W, P)) < 0.8)          # some empty partitions
    bufs = [dict() for _ in range(W)]
    totals = None
    for me in range(W):
        pos, send, recv, local = cgd.exchange_plan(P, W, me, counts)
        pos_begin, total, adj = cgd.peer_plan(P, W, me, counts)
        totals = total if totals is None else totals
        assert np.array_equal(total, totals)                       # every rank computes the same strides
        order = np.argsort(pos)
        i = 0
        for q in range(P):
            p = int(order[q])
            d = int(np.searchsorted(pos_begin, q, side="right") - 1)
            assert d == p % W
            for k in range(int(counts[me, p])):
                at = int(adj[d]) + i
                assert at not in bufs[d]
                bufs[d][at] = (me, p, k)
                i += 1
        assert i == int(send.sum())
    for d in range(W):
        parts = [p for p in range(P) if p % W == d]
        want = [(r, p, k) for r in range(W) for p in parts for k in range(int(counts[r, p]))]
        assert int(totals[d]) == len(want) and sorted(bufs[d]) == list(range(len(want)))
        assert [bufs[d][i] for i in range(len(want))] == want


# --------------------------------------------------------------------------- lane-per-stream LZ4 decoder (on the host)
@pytest.fixture(scope="module")
def lz4_lane_host():
    """tests/helpers/lz4_lane_host.cpp: the decoder source of cg_lz4_lane_kernel compiled for the host (g++), a
    test-only shared object -- libcitus_gpu.so itself has no host decoding path"""
    import subprocess
    out_dir = os.path.join(ROOT, "tests", "helpers", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "liblz4_lane_host.so")
    src = os.path.join(ROOT, "tests", "helpers", "lz4_lane_host.cpp")
    hdr = os.path.join(ROOT, "citus_b200", "csrc", "cg_lz4_lane.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["g++", "-O2", "-g", "-shared", "-fPIC", "-x", "c++", "-I", os.path.dirname(hdr), "-o", so, src])
    L = C.CDLL(so)
    L.lz4_lane_decode_host.restype = C.c_int
    L.lz4_lane_decode_host.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_uint, C.c_uint, C.c_uint]
    return L


def _lz4_lane_decode(lib, comp, rawlen, lane=0, slack=48):
    padded = (rawlen + 15) // 16 * 16 + 16
    src = np.frombuffer(bytes(comp) + bytes(16), np.uint8).copy()
    dst = np.full(padded + slack, 0xEE, np.uint8)
    ok = lib.lz4_lane_decode_host(src.ctypes.data, len(comp), dst.ctypes.data, rawlen, padded, lane)
    assert (dst[padded:] == 0xEE).all(), "wrote past the slot"
    return ok, dst[:padded]


def test_lz4_lane_decoder_against_liblz4(oracle, lz4_lane_host):
    """cg_lz4_lane.cuh is sequential code one GPU lane runs per value stream; the same source is executed here against
    streams produced by liblz4's LZ4_compress_default (what the reference's CompressBuffer calls): literal runs and
    matches of every length class, offsets inside and beyond the 2 KB window, overlapping matches, stream sizes around
    the window / piece / 16-byte flush boundaries; truncated and damaged streams are rejected or decode to the wrong
    bytes of the right size only where liblz4 itself would"""
    if not oracle.lib().orc_have_lz4():
        pytest.skip("liblz4 missing")
    rng = np.random.default_rng(5)
    cases = {
        "empty": b"", "one byte": b"x", "15 bytes": bytes(range(15)), "zeros 100k": bytes(100_000),
        "period 3": (b"abc" * 40_000)[:100_000], "period 1021 (beyond the window)": bytes(rng.integers(0, 256, 1021, dtype=np.uint8)) * 90,
        "period 1024": bytes(rng.integers(0, 256, 1024, dtype=np.uint8)) * 90,
        **{f"period {p} (around the window's reach)": bytes(rng.integers(0, 256, p, dtype=np.uint8)) * 40 for p in (1999, 2000, 2001, 2047, 2048, 2049)},
        "period 5000": bytes(rng.integers(0, 256, 5000, dtype=np.uint8)) * 20,
        "period 60000 (max offsets)": bytes(rng.integers(0, 256, 60_000, dtype=np.uint8)) * 3,
        "C2 key column": rng.integers(0, 10**6, 10_000).astype(np.int64).tobytes(),
        "C2 f column": rng.integers(0, 100, 10_000).astype(np.int64).tobytes(),
        "C2 v column": rng.integers(-10**9, 10**9, 10_000).astype(np.int64).tobytes(),
        "int4 dates": rng.integers(-2922, -365, 10_000).astype(np.int32).tobytes(),
        "incompressible": rng.integers(0, 256, 80_000).astype(np.uint8).tobytes(),
        "text": (b"the quick brown fox jumps over the lazy dog. " * 3000)[:100_000],
        "runs": np.repeat(rng.integers(0, 100, 200), 500).astype(np.int8).tobytes(),
        "sorted ids": np.arange(10_000, dtype=np.int64).tobytes(),
    }
    for n in (2, 3, 12, 13, 16, 17, 31, 255, 256, 257, 270, 271, 272, 1008, 1023, 1024, 1025, 1039, 1040, 1041, 1279, 1280, 1281, 2000, 2047, 2048, 2049, 2063, 2064, 2065, 2303, 2304,
              4095, 4096, 65_535, 65_536, 65_537, 80_000):
        cases[f"mixed n={n}"] = (rng.integers(0, 50, n) * rng.integers(0, 2, n)).astype(np.uint8).tobytes()
        cases[f"sparse n={n}"] = (rng.integers(0, 256, n) * (rng.integers(0, 40, n) == 0)).astype(np.uint8).tobytes()
    for name, data in cases.items():
        comp = oracle.codec_compress(oracle.COMP_LZ4, data, 0)
        assert comp is not None
        for lane in (0, 7, 31):
            ok, out = _lz4_lane_decode(lz4_lane_host, comp, len(data), lane)
            assert ok == 1 and out[:len(data)].tobytes() == data and not out[len(data):].any(), (name, lane)
        # a truncated stream never decodes to the full size; a wrong expected size is refused
        if len(comp) > 1:
            ok, _ = _lz4_lane_decode(lz4_lane_host, comp[:-1], len(data))
            assert ok == 0, (name, "truncated")
        ok, _ = _lz4_lane_decode(lz4_lane_host, comp, len(data) + 1)
        assert ok == 0, (name, "one byte more expected")
        if len(data) > 0:
            ok, _ = _lz4_lane_decode(lz4_lane_host, comp, len(data) - 1)
            assert ok == 0, (name, "one byte less expected")
    # damaged streams: whatever happens stays inside the slot (checked by _lz4_lane_decode) and agrees with liblz4
    for name in ("C2 key column", "text", "period 5000", "mixed n=4096"):
        data = cases[name]
        comp = bytearray(oracle.codec_compress(oracle.COMP_LZ4, data, 0))
        for _ in range(300):
            bad = bytearray(comp)
            for _ in range(int(rng.integers(1, 4))):
                bad[int(rng.integers(0, len(bad)))] = int(rng.integers(0, 256))
            ok, out = _lz4_lane_decode(lz4_lane_host, bytes(bad), len(data))
            try:
                ref = oracle.codec_decompress(oracle.COMP_LZ4, bytes(bad), len(data))
            except oracle.OracleError:
                ref = None
            if ok == -1:
                continue        # a match with offset 0: refused here; liblz4 copies what the output buffer held before
            assert (ok == 1) == (ref is not None), name
            if ok == 1:
                assert out[:len(data)].tobytes() == ref, name


def test_lz4_lane_hand_assembled_blocks(lz4_lane_host):
    """known-answer blocks: the golden of tests/test_oracle_golden.py, maximum-length codes, offset == position"""
    # [token: 1 literal | match 10-4]['a'][offset 1] [token: 5 literals]['aaaaa'] -> 16 x 'a'
    blk = bytes([0x16, ord("a"), 1, 0, 0x50]) + b"aaaaa"
    ok, out = _lz4_lane_decode(lz4_lane_host, blk, 16)
    assert ok == 1 and out[:16].tobytes() == b"a" * 16
    # literal length 15 + 255 + 3 = 273 and a match of 4 + 15 + 255 + 255 + 7 = 536 bytes at offset 273 (the whole prefix), then 5 literals
    lits = bytes((i * 7) & 0xff for i in range(273))
    blk = bytes([0xFF, 255, 3]) + lits + bytes([273 & 0xff, 273 >> 8, 255, 255, 7]) + bytes([0x50]) + b"vwxyz"
    want = lits + (lits * 2)[:536] + b"vwxyz"
    ok, out = _lz4_lane_decode(lz4_lane_host, blk, len(want))
    assert ok == 1 and out[:len(want)].tobytes() == want
    # offset 0, offset beyond the output, match past the expected size, literals past the stream: all refused
    for bad, raw in ((bytes([0x10, 1, 0, 0, 0x00]), 8), (bytes([0x10, 1, 2, 0, 0x00]), 8), (bytes([0x1F, 1, 1, 0, 200, 0x00]), 20),
                     (bytes([0x50, 1, 2]), 5), (b"", 0)):
        ok, _ = _lz4_lane_decode(lz4_lane_host, bad, raw)
        assert ok != 1
    # an empty output is exactly the one-byte block [0] (liblz4's rule)
    assert _lz4_lane_decode(lz4_lane_host, bytes([0]), 0)[0] == 1 and _lz4_lane_decode(lz4_lane_host, bytes([0x03]), 0)[0] != 1


# --------------------------------------------------------------------------- Zstandard decoder (format logic on the host)
@pytest.fixture(scope="module")
def zstd_host():
    """tests/helpers/zstd_host.cpp: the decoder source of the GPU kernel compiled for the host (g++), a test-only
    shared object -- libcitus_gpu.so itself has no host decoding path"""
    import subprocess
    out_dir = os.path.join(ROOT, "tests", "helpers", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libzstd_host.so")
    src = os.path.join(ROOT, "tests", "helpers", "zstd_host.cpp")
    hdr = os.path.join(ROOT, "citus_b200", "csrc", "cg_zstd.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", "-I", os.path.dirname(hdr), "-o", so, src])
    L = C.CDLL(so)
    L.zstd_decode_host.restype = C.c_longlong
    L.zstd_decode_host.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_uint]
    return L


def test_zstd_decoder_against_libzstd(cg, oracle, zstd_host):
    """cg_zstd.cuh is sequential code one GPU lane runs; the same source is executed here on the host
    against streams produced by libzstd's ZSTD_compress (what the reference's CompressBuffer calls)"""
    from citus_b200 import capi
    if not oracle.lib().orc_have_zstd():
        pytest.skip("libzstd missing")
    rng = np.random.default_rng(0)
    cases = {
        "empty": b"", "one byte": b"x", "zeros": bytes(100_000),
        "arange%7 int64": (np.arange(10_000) % 7).astype(np.int64).tobytes(),
        "uniform<100 int64": rng.integers(0, 100, 10_000).astype(np.int64).tobytes(),
        "uniform<1e6 int64": rng.integers(0, 10**6, 10_000).astype(np.int64).tobytes(),
        "incompressible": rng.integers(0, 256, 80_000).astype(np.uint8).tobytes(),          # raw blocks
        "signed int64": rng.integers(-10**9, 10**9, 10_000).astype(np.int64).tobytes(),
        "text": (b"the quick brown fox jumps over the lazy dog. " * 3000)[:100_000],
        "800 KB, several blocks": rng.integers(0, 1000, 100_000).astype(np.int64).tobytes(),  # repeat modes / treeless literals
        "skewed bytes": rng.choice(np.arange(256, dtype=np.uint8), 200_000, p=np.r_[0.5, np.full(255, 0.5 / 255)]).tobytes(),
        "runs": np.repeat(rng.integers(0, 100, 200), 500).astype(np.int8).tobytes(),         # RLE blocks / long matches
    }
    for n in (2, 3, 17, 255, 256, 257, 4095, 65_536, 131_071, 131_072, 131_073, 262_145):
        cases[f"mixed n={n}"] = (rng.integers(0, 50, n) * rng.integers(0, 2, n)).astype(np.uint8).tobytes()
    for name, data in cases.items():
        for level in ((1, 3, 9, 19) if len(data) <= 200_000 and not name.startswith("mixed") else (3,)):
            comp = oracle.codec_compress(oracle.COMP_ZSTD, data, level)
            assert comp is not None
            src = np.frombuffer(comp, np.uint8)
            dst = np.zeros(len(data) + 64, np.uint8)
            n = zstd_host.zstd_decode_host(src.ctypes.data, len(comp), dst.ctypes.data, len(data))
            assert n == len(data) and dst[:len(data)].tobytes() == data, (name, level)
            # damaged streams are rejected, never decoded to something else of the right size silently ... except
            # where the damage lands in unused bits; a truncated stream always fails
            if len(comp) > 12:
                n = zstd_host.zstd_decode_host(src.ctypes.data, len(comp) - 1, dst.ctypes.data, len(data))
                assert n != len(data), (name, level, "truncated")


def test_zstd_hand_assembled_frames(cg, oracle, zstd_host):
    """frames built by hand from RFC 8878 (no encoder involved): a raw block, an RLE block, two blocks,
    and malformed variants; the library's decoder and libzstd (through the oracle) must agree"""
    from citus_b200 import capi

    def frame(blocks, fcs):
        out = bytes([0x28, 0xB5, 0x2F, 0xFD, 0x20, fcs])            # magic, FHD: single segment + 1-byte content size
        for i, (btype, size, payload) in enumerate(blocks):
            hdr = (size << 3) | (btype << 1) | (1 if i == len(blocks) - 1 else 0)
            out += hdr.to_bytes(3, "little") + payload
        return out

    def ours(data, cap):
        src = np.frombuffer(data, np.uint8)
        dst = np.zeros(cap + 8, np.uint8)
        n = zstd_host.zstd_decode_host(src.ctypes.data, len(data), dst.ctypes.data, cap)
        return n, dst[:max(n, 0)].tobytes()

    cases = [
        (frame([(0, 5, b"hello")], 5), b"hello"),
        (frame([(1, 7, b"z")], 7), b"z" * 7),
        (frame([(0, 3, b"abc"), (1, 4, b"!")], 7), b"abc!!!!"),
    ]
    for data, want in cases:
        n, got = ours(data, len(want))
        assert n == len(want) and got == want
        if oracle.lib().orc_have_zstd():
            assert oracle.codec_decompress(oracle.COMP_ZSTD, data, len(want)) == want
    bad = [
        frame([(0, 5, b"hello")], 6),                                   # content size does not match
        frame([(3, 5, b"hello")], 5),                                   # reserved block type
        frame([(0, 5, b"hell")], 5),                                    # truncated
        b"\x28\xB5\x2F\xFE" + frame([(0, 5, b"hello")], 5)[4:],         # wrong magic
        frame([(0, 5, b"hello")], 5) + b"x",                            # trailing garbage
    ]
    for data in bad:
        n, _ = ours(data, 16)
        assert n < 0, data


def test_qual_on_column_added_after_the_stripe_was_written(cg):
    """ALTER TABLE ADD COLUMN: a stripe written with fewer columns than the relation has now has no skip
    nodes for the new column; the reference gives it zeroed nodes without min/max (ReadStripeSkipList,
    columnar_metadata.c:753-760), so a WHERE on that column skips no chunk group -- and must not read
    another stripe's nodes (or past the node array)."""
    from citus_b200 import capi
    rng = np.random.default_rng(3)
    n = 9000
    a = np.arange(n)
    b = rng.integers(0, 100, n)
    rel2 = cg.Relation.write([8, 8], [a, b], stripe_row_limit=3000, chunk_row_limit=1000)
    assert rel2.view.nstripes == 3 and rel2.view.stripes[0].column_count == 2
    rel3 = cg.Relation.from_image(rel2.pages(), rel2.stripes_bytes(), rel2.nodes_bytes(), [8, 8, 8])
    d = cg.make_desc([(2, "<", 5)], [], [cg.count_star()])
    for si in range(3):
        mask = np.zeros(3, np.uint8)
        filtered = C.c_int64(-1)
        capi.check(capi.lib().cg_selected_chunk_mask(C.byref(rel3.view), si, C.byref(d), mask.ctypes.data, C.byref(filtered)))
        assert mask.tolist() == [1, 1, 1] and filtered.value == 0
    # a qual on an existing column still skips: a >= 8000 leaves only the last chunk of the last stripe
    d = cg.make_desc([(0, ">=", 8000), (2, "<", 5)], [], [cg.count_star()])
    total = 0
    for si in range(3):
        mask = np.zeros(3, np.uint8)
        filtered = C.c_int64(-1)
        capi.check(capi.lib().cg_selected_chunk_mask(C.byref(rel3.view), si, C.byref(d), mask.ctypes.data, C.byref(filtered)))
        total += filtered.value
    assert total == 8


def test_where_tree_chunk_mask_matches_reference_goldens(cg, expected):
    """SelectedChunkMask over OR / AND trees on the host (cg_selected_chunk_mask): the pushdown_test goldens of
    expected/columnar_chunk_filtering.out; malformed trees are refused"""
    from citus_b200 import capi
    a = np.arange(1, 200001)
    rel = cg.Relation.write([4, 4], [a, np.zeros_like(a)], [None, np.ones(a.shape[0], np.uint8)],
                            stripe_row_limit=2000, chunk_row_limit=1000)
    trees = {
        "a = 204356 or a = 104356 or a = 76556": ("or", (0, "=", 204356), (0, "=", 104356), (0, "=", 76556)),
        "a = 194356 or a = 104356 or a = 76556": ("or", (0, "=", 194356), (0, "=", 104356), (0, "=", 76556)),
        "(a > 1000 and a < 10000) or (a > 20000 and a < 50000)":
            ("or", ("and", (0, ">", 1000), (0, "<", 10000)), ("and", (0, ">", 20000), (0, "<", 50000))),
    }
    for g in expected["pushdown_or"]:
        d = cg.make_desc(trees[g["where"]], [], [cg.sum_(0)])
        total = 0
        for si in range(rel.view.nstripes):
            mask = np.zeros(rel.view.stripes[si].chunk_count, np.uint8)
            f = C.c_int64()
            capi.check(capi.lib().cg_selected_chunk_mask(C.byref(rel.view), si, C.byref(d), mask.ctypes.data, C.byref(f)))
            total += f.value
        assert total == g["groups_removed"]
    d = cg.make_desc(("or", (0, "=", 1), (0, "=", 2)), [], [cg.count_star()])
    d.qual_expr[2] = 5                         # refers to an atom that does not exist
    kmin, kmax, rows = C.c_int64(), C.c_int64(), C.c_int64()
    bounds = (C.c_int64 * 8)()
    kind = C.c_int32()
    cols = (capi.CgColumnDesc * 2)()
    cols[0].attlen = cols[1].attlen = 4
    assert capi.lib().cg_jit_compile_check(C.byref(d), cols, 2, 0, -1, 10, C.byref(kind), None, 0) == capi.CG_EINVAL
    d = cg.make_desc(("or", (0, "=", 1), (0, "=", 2)), [], [cg.count_star()])
    d.nqual_expr = 2                           # operands left on the stack
    assert capi.lib().cg_jit_compile_check(C.byref(d), cols, 2, 0, -1, 10, C.byref(kind), None, 0) == capi.CG_EINVAL


def _jit_check_nullable(cg, quals, group, aggs, lens, kmin, kmax, rows, nullable, float_cols=()):
    from citus_b200 import capi
    d = cg.make_desc(quals, group, aggs, float_cols=float_cols)
    cols = (capi.CgColumnDesc * len(lens))()
    for i, l in enumerate(lens):
        cols[i].attlen, cols[i].type_class = l, (1 if i in float_cols else 0)
    kind = C.c_int32(-1)
    buf = C.create_string_buffer(1 << 19)
    rc = capi.lib().cg_jit_compile_check_nullable(C.byref(d), cols, len(lens), kmin, kmax, rows, nullable, C.byref(kind), buf, len(buf))
    assert rc == 0, capi.lib().cg_last_error().decode()
    return kind.value, buf.value.decode()


def test_jit_nullable_and_where_tree_forms_compile(cg):
    """the generated kernels' NULL-aware form (exists bitmap + rank directory, columnar_reader.c:1506-1572) and
    WHERE trees, for every table kind and column width"""
    try:
        C.CDLL("libnvrtc.so.12")
    except OSError:
        pytest.skip("libnvrtc missing")
    a = [cg.sum_(2), cg.count_star()]
    a[0].term_abs_bound = 10**9
    # C2 with NULLs in v: packed word gets count only for a NULL input, the NULL-input counter one more reduction
    kind, src = _jit_check_nullable(cg, [(1, "<", 50)], [0], a, [8] * 8, 0, 999_999, 10**9, 0b100)
    assert kind == 2 and "__popcll(bw" in src and "an0 ? 0ull" in src and "const bool n2" in src and "const bool n0" not in src
    # every column nullable: NULL key -> the entry behind the table, NULL qual input -> atom not TRUE
    kind, src = _jit_check_nullable(cg, [(1, "<", 50)], [0], a, [8] * 8, 0, 999_999, 10**9, 0b111)
    assert "z1 ? P.capacity" in src and "!z0 && " in src
    # hash table, OR tree with an AND arm, count(x), min, narrow columns
    kind, src = _jit_check_nullable(cg, ("or", (1, "<", 50), ("and", (3, ">", 5), (3, "<", 9))), [0],
                                    a + [cg.count(3), cg.min_(4)], [8, 8, 8, 4, 2, 1], 0, -1, 10**9, 0b111111)
    assert kind == 2 and "(t0 || (t1 && t2))" in src and "ld4(" in src and "ld2(" in src
    # plain aggregate: NULL-input counters in registers
    kind, src = _jit_check_nullable(cg, [(1, "<", 50)], [], [cg.sum_(2), cg.count_star(), cg.count(3), cg.min_(4), cg.max_(5)],
                                    [8, 4, 2, 1, 8, 8], 0, -1, 10**9, 0b111111)
    assert kind == 0 and "g_n2++" in src and "ld1(" in src
    # Q1 shape with NULLs everywhere: shared-memory cells, NULL multi-key is flagged
    q1 = [cg.sum_(0), cg.sum_(1), cg.Agg(2, [(1, 0, 1), (2, 100, -1)]), cg.Agg(2, [(1, 0, 1), (2, 100, -1), (3, 100, 1)]),
          cg.sum_(2), cg.count_star()]
    for x, b in zip(q1, (5100, 10_500_000, 10**9, 2 * 10**11, 11, 0)):
        x.term_abs_bound = b
    kind, src = _jit_check_nullable(cg, [(6, "<=", -486)], [4, 5], q1, [8, 8, 8, 8, 1, 1, 4, 4], 65 | (70 << 32), 67 | (71 << 32),
                                    6 * 10**8, 0xff)
    assert kind == 1 and "raise_flag(P.stats, 2ull)" in src
    # one nullable group column on shared-memory cells: the NULL group goes to its global entry
    kind, src = _jit_check_nullable(cg, [(6, "<=", -486)], [4], q1, [8, 8, 8, 8, 1, 1, 4, 4], 65, 67, 6 * 10**8, 0xff)
    assert kind == 1 and "P.table + P.capacity *" in src
    # float columns
    kind, src = _jit_check_nullable(cg, [(1, "<", 0.5)], [0], [cg.sum_(1, True), cg.min_(2, True), cg.count_star()], [8, 8, 4], 0, -1,
                                    10**6, 0b111, float_cols=(1, 2))
    assert kind == 2 and "fcmp(" in src
