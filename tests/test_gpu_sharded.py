"""GPU test of the dimension-sharded search on ONE device: two ranks run as two host threads with their own contexts, the two
collectives are implemented by the test through host memory.  The result must equal the single-rank search bit for bit."""
import ctypes as C
import threading

import numpy as np
import pytest

from golden_util import _random_problem, search_problem

pytestmark = pytest.mark.gpu


class ThreadCollectives:
    """abw_collectives for `world` threads of one process (device buffers are staged through numpy)."""

    def __init__(self, ctxs):
        from abawaca_b200 import capi
        self.world = len(ctxs)
        self.barrier = threading.Barrier(self.world)
        self.slots = [None] * self.world
        self.structs, self._keep = [], []
        for rank, ctx in enumerate(ctxs):
            def allgather(user, d_send, d_recv, nbytes, rank=rank, ctx=ctx):
                buf = np.empty(nbytes, dtype=np.uint8)
                ctx.to_host(buf, d_send)
                self.slots[rank] = buf
                self.barrier.wait()
                ctx.to_device(d_recv, np.concatenate(self.slots))
                self.barrier.wait()
                return 0

            def allreduce(user, d_buf, count, rank=rank, ctx=ctx):
                buf = np.empty(count, dtype=np.int64)
                ctx.to_host(buf, d_buf)
                self.slots[rank] = buf
                self.barrier.wait()
                ctx.to_device(d_buf, np.sum(self.slots, axis=0, dtype=np.int64))
                self.barrier.wait()
                return 0
            ag, ar = capi.ALLGATHER_FN(allgather), capi.ALLREDUCE_FN(allreduce)
            self._keep += [ag, ar]
            st = capi.Collectives(ag, ar, None, rank, self.world)
            self.structs.append(type("S", (), {"struct": st})())


def _problem(name):
    """A golden set, or "random_w3": a generated problem whose SCG masks have three words (160 names, contamination across centres, dense scaffolds)."""
    if name == "random_w3":
        vals, dp2scaf, T, length, mask = _random_problem(np.random.default_rng(41), 1500, 6, ties=False, nclus=5, G=160, contamination=0.001, dense=6)
        assert mask.shape[1] == 3 and mask[:, 2].any()
        return {"values": vals, "dp2scaf": dp2scaf, "T": T, "len": length, "scgmask": mask}
    return search_problem(name)


@pytest.mark.parametrize("name,strategy,world,strided", [("tiny_noisy", 0, 2, False), ("tiny_noisy", 1, 2, False), ("tiny_clean", 0, 3, False),
                                                         ("tiny_noisy", 0, 3, True), ("tiny_clean", 1, 2, True), ("random_w3", 0, 3, True)])
def test_sharded_search_equals_single_rank(name, strategy, world, strided):
    from abawaca_b200 import capi, pipeline, distributed
    prob = _problem(name)
    vals = prob["values"]
    D = vals.shape[0]
    p = capi.default_params()
    p.min_reported_score = 0.0
    ctx0 = capi.Context(0)
    ref = pipeline.search(ctx0, vals, prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], params=p, strategy=strategy)
    ctx0.close()
    assert len(ref.recs) > 1                            # the search splits: there are child clusters to compare
    ctxs = [capi.Context(0) for _ in range(world)]
    coll = ThreadCollectives(ctxs)
    results, errors = [None] * world, []

    def run(rank):
        try:
            if strided:                                     # round-robin dimensions: rank r holds r, r + world, ...
                mine, off, stride = np.ascontiguousarray(vals[rank::world]), rank, world
            else:
                off, cnt = distributed.dim_block(D, rank, world)
                mine, stride = np.ascontiguousarray(vals[off:off + cnt]), 1
            results[rank] = pipeline.search(ctxs[rank], mine, prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], params=p,
                                            strategy=strategy, collectives=coll.structs[rank], dim_offset=off, dim_stride=stride, D_total=D)
        except Exception as e:
            errors.append(e)
            coll.barrier.abort()

    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=120)
    assert not errors, errors
    key = lambda r: (r.id, r.parent, r.ndps, r.nscafs, r.split, r.best.found, r.best.dim, r.best.value, r.best.a, r.best.b, r.child1, r.child2, r.child1_ndps,
                     r.child2_ndps, r.child1_nscafs, r.child2_nscafs, r.child1_raw, r.child2_raw, r.total_size, r.scg_unique, r.scg_avg)   # noqa: E731
    for res in results:
        assert [key(r) for r in res.recs] == [key(r) for r in ref.recs]
        assert res.scaf2cluster.tolist() == ref.scaf2cluster.tolist() and res.dp2cluster.tolist() == ref.dp2cluster.tolist()
    for c in ctxs:
        c.close()


@pytest.fixture()
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def test_column_scatter_kernel_on_one_rank(ctx):
    """abw_scatter_columns_milli with a group of one (no IPC involved): the receiver's matrix holds the integer thousandths of the rows of the scaffolds
    with at least two windows, in order -- what abw_search_create_from_features keeps -- and a search on it equals the search on the doubles.  The split
    of the columns over several ranks is checked by `bench.py --gpus N` (sharded_equals_single) on real peers."""
    import ctypes as C
    from abawaca_b200 import capi, pipeline, synth
    L = ctx.lib
    mg = synth.make_metagenome(1500, 3, 4, 51, min_len=1500, mean_extra=3000)
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0)
    counts = np.diff(fb.seg_first_host().astype(np.int64))
    assert (counts < 2).any()
    keep, dp2scaf, T, kept = pipeline.search_problem_from_counts(counts)
    rows = fb.rows_host()[keep]
    buf, grp, handle = C.c_void_p(), C.c_void_p(), (C.c_ubyte * 64)()
    nbytes = rows.shape[0] * fb.ncols * 4
    ctx.check(L.abw_peer_buffer_create(ctx.h, nbytes + 1024, C.byref(buf), handle))
    ctx.check(L.abw_peer_group_create(ctx.h, buf, bytes(handle), 0, 1, C.byref(grp)))
    flag = ctx.alloc(16)
    ctx.memset(flag, 0, 16)
    ctx.check(L.abw_scatter_columns_milli(ctx.h, grp, fb.segs, C.c_void_p(fb.d_rows), fb.nseg, fb.ncols, fb.ncols, 0, 256, C.c_void_p(flag)))
    got = np.zeros((rows.shape[0], fb.ncols), dtype=np.uint32)
    ctx.to_host(got, buf.value + 256)
    bad = np.zeros(4, dtype=np.int32)
    ctx.to_host(bad, flag)
    assert bad[0] == 0
    assert np.array_equal(got / 1000.0, rows)
    length = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)[kept]
    mask = mg.scg_masks()[kept]
    a = pipeline.search(ctx, buf.value + 256, dp2scaf, T, length, mask, layout=capi.LAYOUT_ROWMAJOR_MILLI32, values_on_device=True, nrows=rows.shape[0], D=fb.ncols, ld=fb.ncols)
    b, _ = pipeline.search_features(ctx, fb, np.diff(mg.offsets.astype(np.int64)).astype(np.uint64), mg.scg_masks())
    assert [(r.id, r.split, r.best.dim, r.best.value) for r in a.recs] == [(r.id, r.split, r.best.dim, r.best.value) for r in b.recs] and len(a.recs) > 1
    assert a.scaf2cluster.tolist() == b.scaf2cluster.tolist()
    # every row (no segments given)
    ctx.check(L.abw_scatter_columns_milli(ctx.h, grp, None, C.c_void_p(fb.d_rows), 100, fb.ncols, fb.ncols, 0, 0, None))
    got = np.zeros((100, fb.ncols), dtype=np.uint32)
    ctx.to_host(got, buf.value)
    assert np.array_equal(got / 1000.0, fb.rows_host()[:100])
    fb.close()
    ctx.free(flag)
    L.abw_peer_group_destroy(grp)
    ctx.check(L.abw_peer_buffer_destroy(ctx.h, buf))
