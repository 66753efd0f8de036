"""The exchange of the sharded search: ctx.finish and ctx.finish_dev accept only the consecutive shards of the plan, in
well-formed partials, and leave the context usable after a rejection; the host partial is the device blob behind a header."""
import numpy as np
import pytest

import asgart_b200 as ab
from tests import cases

pytestmark = pytest.mark.gpu

MAGIC = 0x4132303050415254   # "A200PART"
ST = ab.RunSettings(min_duplication_length=1000, reverse=True, complement=True)


@pytest.fixture(scope="module")
def run():
    """The small text of test_sharded_search_equals_single, indexed once; its single-search families."""
    text = cases.stress_text(12)
    prep = ab.Prepared.from_memory(text, [("a", 0, 25000), ("b", 25000, len(text) - 25000)])
    with ab.Context(0) as ctx:
        ctx.load_strand(np.array(prep.strand))
        ctx.build_index()
        yield ctx, prep.chunks, ctx.search(prep.chunks, ST, ab.POST_ALL).as_lists()


def test_finish_rejects_bad_partials(run):
    ctx, chunks, single = run
    p = [ctx.search_shard(chunks, ST, r, 3) for r in range(3)]
    q = [ctx.search_shard(chunks, ST, r, 2) for r in range(2)]
    other = [ctx.search_shard(chunks[:1], ST, r, 3) for r in range(3)]
    assert ctx.finish(chunks, ST, p, ab.POST_ALL).as_lists() == single
    magic = p[1].copy()
    magic[0] ^= 0xFF
    bad = {
        "out of order": [p[1], p[0], p[2]],
        "middle shard missing": [p[0], p[2]],
        "last shard missing": [p[0], p[1]],
        "shard given twice": [p[0], p[1], p[1], p[2]],
        "2-way and 3-way mixed (overlap)": [q[0], p[1], p[2]],
        "2-way and 3-way mixed (gap)": [p[0], q[1]],
        "cut short by 1 byte": [p[0], p[1][:-1], p[2]],
        "1 byte appended": [p[0], np.concatenate([p[1], np.zeros(1, np.uint8)]), p[2]],
        "flipped magic": [p[0], magic, p[2]],
        "another chunk list": other,
    }
    for label, parts in bad.items():
        with pytest.raises(ab.AsgartB200Error):
            ctx.finish(chunks, ST, parts, ab.POST_ALL)
            pytest.fail(label)
    assert ctx.search(chunks, ST, ab.POST_ALL).as_lists() == single
    assert ctx.finish(chunks, ST, p, ab.POST_ALL).as_lists() == single


def test_finish_dev_rejects_bad_shards(run):
    import torch
    from asgart_b200.dist import _DevMem
    ctx, chunks, single = run
    blobs, metas = [], []   # each blob cloned to torch memory, as an all-gather leaves it
    for r in range(3):
        ptr, nbytes, meta = ctx.search_shard_dev(chunks, ST, r, 3)
        blobs.append(torch.as_tensor(_DevMem(ptr, nbytes), device="cuda:0").clone())
        metas.append(meta)
    torch.cuda.synchronize()
    ptrs = [b.data_ptr() for b in blobs]

    def finish(order, meta_edit=None, null=None):
        m = np.stack([metas[r] for r in order])
        if meta_edit:
            meta_edit(m)
        pp = [0 if r == null else ptrs[r] for r in order]
        return ctx.finish_dev(chunks, ST, pp, m, ab.POST_ALL)

    assert finish([0, 1, 2]).as_lists() == single

    def over_total(m):
        m[-1, 1] += 32

    bad = {
        "out of order": dict(order=[1, 0, 2]),
        "gap": dict(order=[0, 2]),
        "short of the total": dict(order=[0, 1]),
        "past the total": dict(order=[0, 1, 2], meta_edit=over_total),
        "null blob": dict(order=[0, 1, 2], null=1),
    }
    for label, kw in bad.items():
        with pytest.raises(ab.AsgartB200Error):
            finish(**kw)
            pytest.fail(label)
    assert ctx.search(chunks, ST, ab.POST_ALL).as_lists() == single
    assert finish([0, 1, 2]).as_lists() == single


@pytest.mark.parametrize("n_shards", [1, 2, 3, 8])
def test_host_partial_is_device_blob(run, n_shards):
    """After its header {magic, p_begin, p_end, events, matches, blob bytes}, search_shard's partial is, byte for byte,
    the blob search_shard_dev leaves in HBM for the same shard (padding of the processed bits included)."""
    import torch
    from asgart_b200.dist import _DevMem
    ctx, chunks, _ = run
    events = 0
    for r in range(n_shards):
        ptr, nbytes, meta = ctx.search_shard_dev(chunks, ST, r, n_shards)
        part = ctx.search_shard(chunks, ST, r, n_shards)   # leaves the device blob as it is
        blob = torch.as_tensor(_DevMem(ptr, nbytes), device="cuda:0").cpu().numpy() if nbytes else np.zeros(0, np.uint8)
        hdr = part[:48].view(np.uint64)
        assert hdr.tolist() == [MAGIC, *meta.tolist(), nbytes], r
        assert np.array_equal(part[48:], blob), r
        events += int(meta[2])
    assert events > 0
