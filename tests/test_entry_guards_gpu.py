"""The checks every column-taking C entry makes before it runs, the same on a one-GPU context and on a multi-GPU context (one of
ONE GPU runs the whole multi-GPU code path): a null column and a column made by another context are BDF_INVALID, an
expression with too few or too many inputs gets the same message on both, and a multi-GPU context refuses inputs with different chunk
counts (BDF_UNSUPPORTED, plain and fused entries alike) and the operators that move rows between chunks."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LENS = [1000, 300]


@pytest.fixture(scope="module")
def contexts(rdf):
    import torch

    if not torch.cuda.device_count():
        pytest.skip("no GPU")
    ctxs = {"one": rdf.Context(0), "multi": rdf.Context.multi(1)}
    yield ctxs
    for c in ctxs.values():
        c.close()


class Columns:
    """Columns made on one context for one test; free() releases all of them."""

    def __init__(self, rdf, ctx):
        self.N, self.L, self.ctx, self.made = rdf.native, rdf.native.lib(), ctx, []

    def upload(self, np_dtype, lens):
        chunks = [self.N.PrimitiveArray.from_numpy(np.arange(n).astype(np_dtype)) for n in lens]
        h = C.c_void_p()
        assert self.L.bdf_upload(self.ctx.handle, chunks[0].dtype, len(chunks), self.N.make_views(chunks), 0, C.byref(h)) == self.N.OK
        self.made.append(h)
        return h

    def mask(self, col):
        h = C.c_void_p()
        assert self.L.bdf_compare_dev(self.ctx.handle, self.N.GT, col, None, 10.0, C.byref(h)) == self.N.OK
        self.made.append(h)
        return h

    def kinds(self, lens=LENS):
        """One column of every kind an entry takes: f (Float64), m (boolean), u (UInt32 indices)."""
        f = self.upload(np.float64, lens)
        return {"f": f, "m": self.mask(f), "u": self.upload(np.uint32, lens)}

    def free(self):
        for h in self.made:
            self.L.bdf_col_free(self.ctx.handle, h)
        self.made = []


def _entries(N, L):
    """name -> (column kinds, call(ctx, *columns) -> status).  Every output a call could make is a throw-away local."""
    out, fut, agg, agg2 = C.c_void_p(), C.c_void_p(), N.Agg4(), (N.Agg4 * 2)()
    scalar, some, dbl, i64, i32 = C.c_uint64(), C.c_int32(), C.c_double(), C.c_int64(), C.c_int32()
    nodes = (N.ExprNode * 1)(N.ExprNode(N.ADD, 0, 1))
    outs = (N.Out * len(LENS))()
    groups, n_groups = N.GroupOut(), C.c_int64()
    r = C.byref

    def arr(*cols):
        return (C.c_void_p * len(cols))(*cols)

    return {
        "binary_dev": ("ff", lambda c, x, y: L.bdf_binary_dev(c, N.ADD, x, y, r(out))),
        "binary_agg_dev": ("ff", lambda c, x, y: L.bdf_binary_agg_dev(c, N.ADD, x, y, r(out), r(agg))),
        "binary_agg_dev_async": ("ff", lambda c, x, y: L.bdf_binary_agg_dev_async(c, N.ADD, x, y, r(out), r(fut))),
        "unary_dev": ("f", lambda c, x: L.bdf_unary_dev(c, N.SIN, x, r(out))),
        "cast_dev": ("f", lambda c, x: L.bdf_cast_dev(c, 8, x, r(out))),
        "aggregate_dev": ("f", lambda c, x: L.bdf_aggregate_dev(c, N.SUM, x, r(scalar), r(some))),
        "aggregate_all_dev": ("f", lambda c, x: L.bdf_aggregate_all_dev(c, x, r(agg))),
        "aggregate_all_dev_async": ("f", lambda c, x: L.bdf_aggregate_all_dev_async(c, x, r(fut))),
        "aggregate_all_many_dev": ("ff", lambda c, x, y: L.bdf_aggregate_all_many_dev(c, 2, arr(x, y), agg2)),
        "aggregate_all_many_dev_async": ("ff", lambda c, x, y: L.bdf_aggregate_all_many_dev_async(c, 2, arr(x, y), r(fut))),
        "avg_dev": ("f", lambda c, x: L.bdf_avg_dev(c, x, r(dbl), r(some))),
        "eval_expr_dev": ("ff", lambda c, x, y: L.bdf_eval_expr_dev(c, 2, arr(x, y), 1, nodes, r(out))),
        "eval_expr_agg_dev": ("ff", lambda c, x, y: L.bdf_eval_expr_agg_dev(c, 2, arr(x, y), 1, nodes, r(out), r(agg))),
        "eval_expr_agg_dev_async": ("ff", lambda c, x, y: L.bdf_eval_expr_agg_dev_async(c, 2, arr(x, y), 1, nodes, r(out), r(fut))),
        "compare_dev": ("ff", lambda c, x, y: L.bdf_compare_dev(c, N.GT, x, y, 0.0, r(out))),
        "boolean_dev": ("mm", lambda c, x, y: L.bdf_boolean_dev(c, N.AND, x, y, r(out))),
        "filter_dev": ("fm", lambda c, x, y: L.bdf_filter_dev(c, x, y, r(out))),
        "take_dev": ("fu", lambda c, x, y: L.bdf_take_dev(c, x, y, r(out))),
        "sort_indices_dev": ("f", lambda c, x: L.bdf_sort_indices_dev(c, 1, (N.SortKeyC * 1)(N.SortKeyC(x, 0)), r(out))),
        "group_aggregate_dev": ("ff", lambda c, x, y: L.bdf_group_aggregate_dev(c, x, 1, arr(y), r(out), r(groups), r(n_groups))),
        "col_wait": ("f", lambda c, x: L.bdf_col_wait(c, x)),
        "col_chunk_info": ("f", lambda c, x: L.bdf_col_chunk_info(c, x, 0, r(i64), r(i64), r(i32))),
        "download": ("f", lambda c, x: L.bdf_download(c, x, outs)),
        "download_begin": ("f", lambda c, x: L.bdf_download_begin(c, x, outs)),
        "download_end": ("f", lambda c, x: L.bdf_download_end(c, x, outs)),
    }


ENTRY_SLOTS = [(name, slot) for name, n in [
    ("binary_dev", 2), ("binary_agg_dev", 2), ("binary_agg_dev_async", 2), ("unary_dev", 1), ("cast_dev", 1), ("aggregate_dev", 1),
    ("aggregate_all_dev", 1), ("aggregate_all_dev_async", 1), ("aggregate_all_many_dev", 2), ("aggregate_all_many_dev_async", 2),
    ("avg_dev", 1), ("eval_expr_dev", 2), ("eval_expr_agg_dev", 2), ("eval_expr_agg_dev_async", 2), ("compare_dev", 2),
    ("boolean_dev", 2), ("filter_dev", 2), ("take_dev", 2), ("sort_indices_dev", 1), ("group_aggregate_dev", 2), ("col_wait", 1),
    ("col_chunk_info", 1), ("download", 1), ("download_begin", 1), ("download_end", 1)] for slot in range(n)]


def _call_with(rdf, ctx, name, slot, column):
    """The entry on ctx with its own valid columns except `column` in argument slot `slot`."""
    N = rdf.native
    kinds, call = _entries(N, N.lib())[name]
    own = Columns(rdf, ctx)
    try:
        cols = own.kinds()
        args = [cols[k] for k in kinds]
        args[slot] = column(kinds[slot])
        return call(ctx.handle, *args)
    finally:
        own.free()


@pytest.mark.parametrize("which", ["one", "multi"])
@pytest.mark.parametrize("name,slot", [e for e in ENTRY_SLOTS if e not in (("compare_dev", 1), ("boolean_dev", 1))])   # optional right sides
def test_null_column_is_invalid(rdf, contexts, which, name, slot):
    assert _call_with(rdf, contexts[which], name, slot, lambda kind: None) == rdf.native.INVALID


@pytest.mark.parametrize("which", ["one", "multi"])
@pytest.mark.parametrize("name,slot", ENTRY_SLOTS)
def test_column_of_another_context_is_invalid(rdf, contexts, which, name, slot):
    other = Columns(rdf, contexts["multi" if which == "one" else "one"])
    try:
        foreign = other.kinds()
        assert _call_with(rdf, contexts[which], name, slot, lambda kind: foreign[kind]) == rdf.native.INVALID
        assert "context that made it" in rdf.native.lib().bdf_last_error().decode()
    finally:
        other.free()


@pytest.mark.parametrize("n_inputs", [0, 9])
def test_expression_input_count_is_checked_alike(rdf, contexts, n_inputs):
    N = rdf.native
    L = N.lib()
    nodes = (N.ExprNode * 1)(N.ExprNode(N.ADD, 0, 1))
    seen = []
    for ctx in contexts.values():
        own = Columns(rdf, ctx)
        try:
            f = own.upload(np.float64, LENS)
            inputs = (C.c_void_p * 9)(*([f] * 9))
            out, fut, agg = C.c_void_p(), C.c_void_p(), N.Agg4()
            for call in (lambda: L.bdf_eval_expr_dev(ctx.handle, n_inputs, inputs, 1, nodes, C.byref(out)),
                         lambda: L.bdf_eval_expr_agg_dev(ctx.handle, n_inputs, inputs, 1, nodes, C.byref(out), C.byref(agg)),
                         lambda: L.bdf_eval_expr_agg_dev_async(ctx.handle, n_inputs, inputs, 1, nodes, C.byref(out), C.byref(fut))):
                assert call() == N.INVALID
                seen.append(L.bdf_last_error().decode())
        finally:
            own.free()
    assert len(set(seen)) == 1 and "input columns" in seen[0], seen


@pytest.mark.parametrize("name", ["binary_dev", "binary_agg_dev", "binary_agg_dev_async", "eval_expr_dev", "eval_expr_agg_dev",
                                  "eval_expr_agg_dev_async", "compare_dev", "boolean_dev"])
def test_multi_gpu_inputs_with_different_chunk_counts_are_unsupported(rdf, contexts, name):
    N = rdf.native
    kinds, call = _entries(N, N.lib())[name]
    own = Columns(rdf, contexts["multi"])
    try:
        a, b = own.kinds([LENS[0]]), own.kinds([LENS[0], 0])   # the same first chunk, one chunk more
        assert call(contexts["multi"].handle, a[kinds[0]], b[kinds[1]]) == N.UNSUPPORTED
    finally:
        own.free()


@pytest.mark.parametrize("name", ["sort_indices_dev", "take_dev", "filter_dev", "group_aggregate_dev"])
def test_multi_gpu_refuses_operators_that_move_rows_between_chunks(rdf, contexts, name):
    N = rdf.native
    kinds, call = _entries(N, N.lib())[name]
    own = Columns(rdf, contexts["multi"])
    try:
        cols = own.kinds()
        assert call(contexts["multi"].handle, *[cols[k] for k in kinds]) == N.UNSUPPORTED
    finally:
        own.free()
