"""The multi-GPU context (bdf_init_multi): ONE process, the library shards every call over the GPUs by row range.
Results must be those of the one-GPU context (bit-exact where the one-GPU path is) for every fleet size, including a
fleet of ONE GPU (which still cuts and re-assembles nothing but runs the whole fleet code path) -- so these tests run on
the one-GPU box too and on 2/4/8 GPUs where the box has them."""
import numpy as np
import pytest

from helpers import assert_same_array

pytestmark = pytest.mark.gpu


def _gpu_count():
    import torch

    return torch.cuda.device_count()


def _sizes():
    """Fleet sizes: 0 (Context.multi's "every visible GPU") and 1 on every machine, so the test ids do not depend on the machine
    that collects them; 2, 3, 4 and 8 where the box has that many GPUs."""
    n = _gpu_count()
    return [0, 1] + [k for k in (2, 3, 4, 8) if k <= n]


def _chunks(rdf, name, seed, lens, null_frac):
    npdt = np.dtype(name)
    rng = np.random.default_rng(seed)
    out = []
    for n in lens:
        if npdt.kind == "f":
            v = rng.uniform(-1e3, 1e3, n).astype(npdt)
        else:
            info = np.iinfo(npdt)
            v = rng.integers(info.min, info.max, n, dtype=npdt, endpoint=True)
        out.append(rdf.PrimitiveArray.from_numpy(v, rng.random(n) >= null_frac if null_frac else None))
    return out


LENS = [100_001, 0, 1, 70_000, 64, 333_333, 4097]


@pytest.fixture(scope="module", params=_sizes())
def fleet(request, rdf):
    n = _gpu_count()
    if not n:
        pytest.skip("no GPU")
    ctx = rdf.Context.multi(request.param)
    assert ctx.n_gpus == (request.param or n)
    yield ctx
    ctx.close()


def test_host_in_host_out_entries_match_the_oracle(rdf, oracle, fleet):
    """The drop-in entries through a fleet: values, validity, null counts and chunk structure as the oracle says."""
    for name, null_frac in [("float64", 0.1), ("int64", 0.2), ("int32", 0.0), ("uint8", 0.3), ("float32", 0.05), ("int16", 0.1)]:
        a, b = _chunks(rdf, name, 1, LENS, null_frac), _chunks(rdf, name, 2, LENS, 0.0 if null_frac < 0.1 else 0.05)
        dtype = a[0].dtype
        for op_name, orc_op in (("add", oracle.ADD), ("multiply", oracle.MUL), ("subtract", oracle.SUB)):
            got = getattr(rdf.ScalarFunctions, op_name)(a, b, ctx=fleet)
            st, want = oracle.col_binary(orc_op, dtype, a, b)
            assert st == oracle.OK and len(got) == len(want)
            for i, (g, w) in enumerate(zip(got, want)):
                assert_same_array(g, w, what=f"{name} {op_name} chunk {i} on {fleet.n_gpus} GPUs")
        agg = rdf.AggregateFunctions.all(a, dtype=dtype, ctx=fleet)
        assert agg["rows"] == sum(LENS) and agg["n_chunks"] == len(LENS) and agg["would_panic"]   # the empty chunk
        assert agg["count"] == int(oracle.aggregate(oracle.COUNT, dtype, a)[1])
        if name.startswith("float"):
            exact, sum_abs = oracle.sum_exact(dtype, a)
            eps = 2.0 ** -53 if name == "float64" else 2.0 ** -24
            assert abs(np.longdouble(agg["sum"]) - exact) <= 16 * np.log2(sum(LENS)) * eps * sum_abs
            got = rdf.ScalarFunctions.sin(a, ctx=fleet)
            st, want = oracle.col_unary(oracle.SIN, dtype, a)
            for i, (g, w) in enumerate(zip(got, want)):
                assert_same_array(g, w, what=f"{name} sin chunk {i}", exact=False, max_ulp=3 if name == "float64" else 5, check_payload=False)
        else:
            nonempty = [c for c in a if c.valid_mask().any()]
            assert int(agg["sum"]) == int(oracle.aggregate(oracle.SUM, dtype, a)[1])
            assert int(agg["min"]) == int(oracle.aggregate(oracle.MIN, dtype, nonempty)[1])
            assert int(agg["max"]) == int(oracle.aggregate(oracle.MAX, dtype, nonempty)[1])
            assert int(rdf.AggregateFunctions.sum(a, dtype=dtype, ctx=fleet)) == int(agg["sum"])
            assert rdf.AggregateFunctions.count(a, dtype=dtype, ctx=fleet) == agg["count"]
            with pytest.raises(rdf.ReferencePanic):
                rdf.AggregateFunctions.max(a, dtype=dtype, ctx=fleet)
            assert int(rdf.AggregateFunctions.max(nonempty, dtype=dtype, ctx=fleet)) == int(agg["max"])
        # cast (fallible for the narrowing ones): values and NULL slots
        to = rdf.F64 if not name.startswith("float") else rdf.I32
        got = rdf.cast(a, to, ctx=fleet)
        st, want = oracle.col_cast(dtype, to, a)
        for i, (g, w) in enumerate(zip(got, want)):
            assert_same_array(g, w, what=f"{name} cast chunk {i}")


def test_an_all_null_piece_is_not_an_all_null_chunk(rdf, oracle, fleet):
    """The reference's max/min panic on a chunk WITHOUT a valid slot.  A fleet cuts chunks into pieces: a piece may be all-null
    while its chunk is not -- the rule must be evaluated over the caller's chunks."""
    n = 64 * 1000 * max(fleet.n_gpus, 2)
    vals = np.arange(n, dtype=np.int64)
    mask = np.zeros(n, dtype=bool)
    mask[:100] = True   # only the first piece holds valid slots
    arr = [rdf.PrimitiveArray.from_numpy(vals, mask)]
    assert int(rdf.AggregateFunctions.max(arr, ctx=fleet)) == 99 and int(rdf.AggregateFunctions.min(arr, ctx=fleet)) == 0
    agg = rdf.AggregateFunctions.all(arr, ctx=fleet)
    assert not agg["would_panic"] and agg["count"] == 100 and int(agg["sum"]) == 99 * 100 // 2


def test_divide_by_zero_and_length_mismatch(rdf, fleet):
    n = 64 * 500 * max(fleet.n_gpus, 1) + 17
    a = [rdf.PrimitiveArray.from_numpy(np.arange(1, n + 1, dtype=np.int32))]
    d = np.full(n, 3, dtype=np.int32)
    d[n - 5] = 0   # the zero sits in the LAST GPU's piece; every GPU must take the same exit
    with pytest.raises(rdf.DivideByZero):
        rdf.ScalarFunctions.divide(a, [rdf.PrimitiveArray.from_numpy(d)], ctx=fleet)
    d[n - 5] = 7
    q = rdf.ScalarFunctions.divide(a, [rdf.PrimitiveArray.from_numpy(d)], ctx=fleet)
    assert np.array_equal(q[0].value_slice(), np.arange(1, n + 1, dtype=np.int32) // d)
    with pytest.raises(rdf.ComputeError):
        rdf.ScalarFunctions.add(a, [rdf.PrimitiveArray.from_numpy(d[:-1])], ctx=fleet)


def test_device_resident_chain_and_fused_entries(rdf, oracle, fleet):
    """Upload once, chain on the devices, download once; fused add+aggregate, multi-column aggregate, fused expression."""
    lens = [250_000, 64, 100_000, 1]
    fa, fb = _chunks(rdf, "float64", 11, lens, 0.0), _chunks(rdf, "float64", 12, lens, 0.1)
    ia, ib = _chunks(rdf, "int64", 13, lens, 0.1), _chunks(rdf, "int64", 14, lens, 0.0)
    ca, cb, ci, cj = rdf.Column.upload_many([fa, fb, ia, ib], ctx=fleet)
    assert ca.n_chunks == len(lens) and len(ca) == sum(lens)
    e = ca.add(cb); g = e.multiply(ca); h = g.sin()
    _, oe = oracle.col_binary(oracle.ADD, oracle.F64, fa, fb)
    _, og = oracle.col_binary(oracle.MUL, oracle.F64, oe, fa)
    _, oh = oracle.col_unary(oracle.SIN, oracle.F64, og)
    for i, (x, w) in enumerate(zip(g.download(), og)):
        assert_same_array(x, w, what=f"chain g chunk {i}")
    for i, (x, w) in enumerate(zip(h.download(), oh)):
        assert_same_array(x, w, what=f"chain h chunk {i}", exact=False, max_ulp=3, check_payload=False)
    assert h.chunk_info(0)["null_count"] == oh[0].null_count
    k, agg = ci.binary_agg(rdf.native.ADD, cj)
    _, ok = oracle.col_binary(oracle.ADD, oracle.I64, ia, ib)
    for key, op in (("sum", oracle.SUM), ("min", oracle.MIN), ("max", oracle.MAX), ("count", oracle.COUNT)):
        assert int(agg[key]) == int(oracle.aggregate(op, oracle.I64, ok)[1]), key
    for i, (x, w) in enumerate(zip(k.download(), ok)):
        assert_same_array(x, w, what=f"fused add chunk {i}")
    many = rdf.Column.aggregate_all_many([ci, ca, cj])
    assert int(many[0]["sum"]) == int(oracle.aggregate(oracle.SUM, oracle.I64, ia)[1]) and int(many[2]["max"]) == int(oracle.aggregate(oracle.MAX, oracle.I64, ib)[1])
    exact, sum_abs = oracle.sum_exact(oracle.F64, fa)
    assert abs(np.longdouble(many[1]["sum"]) - exact) <= 16 * np.log2(sum(lens)) * 2.0 ** -53 * sum_abs
    fut = rdf.Column.aggregate_all_many([ci, cj], asynchronous=True)
    r = fut.result()
    assert int(r[0]["sum"]) == int(many[0]["sum"]) and int(r[1]["min"]) == int(many[2]["min"])
    w, wa = rdf.eval_expr_agg([ca, cb], [(rdf.native.ADD, 0, 1), (rdf.native.MUL, 2, 0)])
    for i, (x, y) in enumerate(zip(w.download(), og)):
        assert_same_array(x, y, what=f"fused expression chunk {i}", check_payload=False)   # null slots of a fused chain carry payload 0
    assert wa["count"] == sum(c.length - c.null_count for c in og)
    m = ca.gt(cb)
    _, om = oracle.compare(oracle.GT, fa[0], fb[0])
    gm = m.download()[0]
    assert np.array_equal(gm.valid_mask(), om.valid_mask()) and np.array_equal(gm.value_bits()[om.valid_mask()], om.value_bits()[om.valid_mask()])
    with pytest.raises(rdf.UnsupportedType):
        ca.filter(m)
    assert int(ci.sum()) == int(many[0]["sum"]) and ci.count() == many[0]["count"]
    avg = ca.avg()
    vals = np.concatenate([c.value_slice() for c in fa])
    assert abs(avg - vals.mean()) <= 1e-9
    for col in (ca, cb, ci, cj, e, g, h, k, w, m):
        col.free()


def test_generated_columns_are_the_same_rows_for_every_fleet_size(rdf, oracle, fleet):
    """bdf_generate on a fleet yields the rows the one-GPU generator yields (so config benchmarks can shard on the device)."""
    lens = [400_000, 123, 400_000]
    col = rdf.Column.generate(rdf.I64, lens, 3, col_id=77, null_mod=10, ctx=fleet)
    got = col.download()
    row = 0
    for i, n in enumerate(lens):
        want = oracle.generate(oracle.I64, 3, 0, 0, 20260924, 77, row, n, 10)
        assert_same_array(got[i], want, what=f"generated chunk {i}")
        row += n
    agg = col.aggregate_all()
    o = [oracle.generate(oracle.I64, 3, 0, 0, 20260924, 77, sum(lens[:i]), n, 10) for i, n in enumerate(lens)]
    for key, op in (("sum", oracle.SUM), ("min", oracle.MIN), ("max", oracle.MAX), ("count", oracle.COUNT)):
        assert int(agg[key]) == int(oracle.aggregate(op, oracle.I64, o)[1]), key
    col.free()


def test_one_context_called_from_several_threads(rdf, oracle, fleet):
    """The reference's callers may sit on different threads (rayon above the function library): calls on one context are
    serialised by the library, results stay those of the oracle."""
    import threading

    lens = [30_000, 0, 64, 12_345]
    work = []
    for t in range(4):
        a, b = _chunks(rdf, "int64", 100 + t, lens, 0.1), _chunks(rdf, "int64", 200 + t, lens, 0.0)
        _, want = oracle.col_binary(oracle.ADD, oracle.I64, a, b)
        nonempty = [c for c in a if c.length]
        work.append((a, b, want, int(oracle.aggregate(oracle.SUM, oracle.I64, nonempty)[1]), nonempty))
    errors = []

    def run(t):
        a, b, want, want_sum, nonempty = work[t]
        try:
            for _ in range(6):
                got = rdf.ScalarFunctions.add(a, b, ctx=fleet)
                for i, (g, w) in enumerate(zip(got, want)):
                    assert_same_array(g, w, what=f"thread {t} chunk {i}")
                assert int(rdf.AggregateFunctions.sum(nonempty, dtype=a[0].dtype, ctx=fleet)) == want_sum
        except BaseException as e:   # noqa: BLE001 -- reported on the main thread
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=run, args=(t,)) for t in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join(timeout=120)
    assert not errors, errors
    assert not any(th.is_alive() for th in threads)
