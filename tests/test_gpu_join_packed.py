"""GPU parity of the fused probe over one-column builds: the packed table ({key, payload} in one 16-byte entry, join.cu PackedSlot) and
the match bitmap every fused probe kernel writes instead of per-row build positions.  Every case is checked against the CPU oracle."""
import numpy as np
import pytest

import oracle_lib as o
from helpers import gpu_join_rows, oracle_join_rows
from trino_b200 import abi
from trino_b200 import operators as ops
from trino_b200.page import Block, Page

pytestmark = pytest.mark.gpu

PAGE_SIZES = [1, 31, 33, 1023, 1024, 1025, 3 * 1024 + 17]
PAYLOADS = {
    "bigint": lambda k: Block.bigint(k * 7 - 1),
    "double": lambda k: Block.double(k * 0.25),
    "integer": lambda k: Block.integer((k % 100_003).astype(np.int32)),
    "smallint": lambda k: Block.smallint((k % 30_011).astype(np.int16)),
    "tinyint": lambda k: Block.tinyint((k % 113).astype(np.int8)),
}


def _build_keys(rng):
    # INT64_MIN is kept beside the table (entry `capacity` of the packed table)
    return np.concatenate([[-2**63], rng.permutation(np.arange(-3000, 40_000)) * 3]).astype(np.int64)


def _probe_pages(rng, okeys, order):
    """one page per size of PAGE_SIZES: about a third of the rows miss, INT64_MIN on the probe side too"""
    pages = []
    for n in PAGE_SIZES:
        k = np.where(rng.random(n) < 0.67, rng.choice(okeys, n), rng.integers(-10_000, 130_000, n)).astype(np.int64)
        k[n // 2] = -2**63
        k = np.sort(k) if order == "ordered" else k
        pages.append(Page(Block.bigint(k), Block.double(k * 0.5)))
    return pages


def _run_device(ctx, build, probe, join_type):
    """one probe page through LookupJoinOperator; returns the output rows and the raw validity bytes of the build column"""
    bridge = ops.JoinBridge()
    b = ops.HashBuilderOperatorFactory(ctx, bridge, [0], [1]).create_operator()
    b.add_input(build)
    b.finish()
    j = ops.LookupJoinOperatorFactory(ctx, bridge, join_type, False, [0], [0, 1]).create_operator()
    j.add_input(probe)
    out = j.get_output_device()
    rows, validity = [], None
    if out is not None:
        col = out.column(2)
        if col.validity:
            validity = ctx.to_host(col.validity, np.uint8, (out.rows + 7) // 8)
        rows = out.to_host().rows()
        out.release()
    j.close()
    b.close()
    bridge.lookup_source.close()
    return rows, validity


@pytest.mark.parametrize("mode", ["0", "1", "2"])
@pytest.mark.parametrize("order", ["ordered", "shuffled"])
@pytest.mark.parametrize("join_type", [abi.JOIN_INNER, abi.JOIN_PROBE_OUTER])
@pytest.mark.parametrize("payload", list(PAYLOADS))
def test_one_column_build_every_payload_width(ctx, monkeypatch, mode, order, join_type, payload):
    """8 / 4 / 2 / 1-byte payloads through the packed table in every table mode, key-ordered and shuffled probe pages of every
    tile shape (whole tiles, ragged tail, both), misses and INT64_MIN on both sides; the index-only positions stay the oracle's."""
    monkeypatch.setenv("TGPU_JOIN_HASH", mode)
    rng = np.random.default_rng([int(mode), len(order), list(PAYLOADS).index(payload)])
    okeys = _build_keys(rng)
    build = Page(Block.bigint(okeys), PAYLOADS[payload](okeys))
    probes = _probe_pages(rng, okeys, order)
    want = []
    for p in probes:
        want.extend(oracle_join_rows(build, p, 0, 0, [0, 1], [1], join_type, False))
    assert gpu_join_rows(ctx, [build], probes, 0, 0, [0, 1], [1], join_type, False) == want
    bridge = ops.JoinBridge()
    b = ops.HashBuilderOperatorFactory(ctx, bridge, [0], [1]).create_operator()
    b.add_input(build)
    b.finish()
    oj = o.Join(build, [0])
    for p in probes:
        keys = Page(p.get_block(0))
        assert (bridge.lookup_source.get_join_positions(keys) == oj.positions(keys, [0])).all()
    oj.close(); b.close(); bridge.lookup_source.close()


@pytest.mark.parametrize("join_type", [abi.JOIN_INNER, abi.JOIN_PROBE_OUTER])
@pytest.mark.parametrize("n", PAGE_SIZES)
@pytest.mark.parametrize("shape", ["no_match", "one_miss", "all_match"])
def test_match_bitmap_is_the_outer_validity(ctx, join_type, n, shape):
    """A PROBE_OUTER page with misses carries the match bitmap as the build column's validity: compared bit for bit (including the
    bits past the last row of a page whose size is not a multiple of 8); a page where every row matches has no validity at all."""
    rng = np.random.default_rng(n)
    okeys = _build_keys(rng)
    build = Page(Block.bigint(okeys), Block.bigint(okeys * 5 + 3))
    if shape == "no_match":
        k = rng.integers(1, 2**40, n) * 3 + 1               # never a multiple of 3: no build key
    else:
        k = rng.choice(okeys, n)
        if shape == "one_miss":
            k[n // 3] = 2**62 + 1
    k = k.astype(np.int64)
    probe = Page(Block.bigint(k), Block.double(k * 0.5))
    rows, validity = _run_device(ctx, build, probe, join_type)
    assert rows == oracle_join_rows(build, probe, 0, 0, [0, 1], [1], join_type, False)
    matched = np.isin(k, okeys)
    if join_type == abi.JOIN_PROBE_OUTER and not matched.all():
        assert validity is not None
        assert (validity == np.packbits(matched, bitorder="little")).all()
    elif rows:
        assert validity is None


@pytest.mark.parametrize("join_type", [abi.JOIN_INNER, abi.JOIN_PROBE_OUTER])
def test_by_reference_host_page_with_misses(ctx, join_type):
    """by-reference host probe pages over a one-column build: INNER drops rows (the other channels are uploaded after all),
    PROBE_OUTER keeps them with NULL build values"""
    rng = np.random.default_rng(17)
    okeys = _build_keys(rng)
    build = Page(Block.bigint(okeys), Block.integer((okeys % 1009).astype(np.int32)))
    probes = []
    for n in (5000, 3 * 1024 + 17):
        k = np.sort(np.where(rng.random(n) < 0.8, rng.choice(okeys, n), rng.integers(-10_000, 130_000, n))).astype(np.int64)
        probes.append(Page(Block.double(rng.normal(size=n)), Block.bigint(k), Block.varchar(["s%d" % i if i % 5 else None for i in range(n)])))
    want = []
    for p in probes:
        want.extend(oracle_join_rows(build, p, 0, 1, [2, 0, 1], [1], join_type, False))
    assert gpu_join_rows(ctx, [build], probes, 0, 1, [2, 0, 1], [1], join_type, False, by_reference=True) == want


@pytest.mark.parametrize("wide", [None, "never"])
@pytest.mark.parametrize("join_type", [abi.JOIN_INNER, abi.JOIN_PROBE_OUTER])
def test_two_column_build_over_key_ordered_page(ctx, monkeypatch, wide, join_type):
    """Two build output columns keep the 16-byte slots + slot-ordered payload arrays (join_probe_lean_kernel) for a key-ordered page;
    TGPU_JOIN_WIDE=never pins that layout, the default reaches it through the locality sampler."""
    if wide:
        monkeypatch.setenv("TGPU_JOIN_WIDE", wide)
    n_orders = 50_000
    okeys = o.synth_orders_keys(n_orders, 0, n_orders, 0x7C02, True)
    lkeys = o.synth_lineitem_keys(n_orders, 0, o.synth_lineitem_rows(n_orders), 0x7C01, False)
    lkeys[::97] += 1                                          # some misses (order keys are sparse: 8 of every 32 values)
    build = Page(Block.bigint(okeys), Block.bigint(okeys % 2557), Block.integer((okeys % 7919).astype(np.int32)))
    probe = Page(Block.bigint(lkeys), Block.double(lkeys * 0.5))
    got = gpu_join_rows(ctx, [build], [probe], 0, 0, [0, 1], [1, 2], join_type, False)
    assert got == oracle_join_rows(build, probe, 0, 0, [0, 1], [1, 2], join_type, False)


def test_one_column_lookup_holds_no_wide_table_and_no_slot_ordered_payload(ctx):
    """tgpu_lookup_memory_bytes: a one-column build adds the payload column and one 16-byte packed entry per slot to the bare
    table; the slot-ordered payload array (8 bytes per slot) and the 32-byte wide slots are gone"""
    n = 200_000
    okeys = np.arange(n, dtype=np.int64) * 4
    sizes = []
    for out in ([], [1]):
        bridge = ops.JoinBridge()
        b = ops.HashBuilderOperatorFactory(ctx, bridge, [0], out).create_operator()
        b.add_input(Page(Block.bigint(okeys), Block.bigint(okeys + 1)))
        b.finish()
        sizes.append(bridge.lookup_source.get_in_memory_size_in_bytes())
        b.close(); bridge.lookup_source.close()
    bare, one_column = sizes
    slots = (bare - n * 8) // 16                              # the bare lookup: 16-byte slots + the key column
    assert slots >= n
    added = one_column - bare - n * 8                         # beyond the payload column itself
    assert (slots + 1) * 16 <= added < (slots + 1) * 16 + 256   # device buffers are allocated in 256-byte units
