"""GPU: HashJoin CUDA path (through the C ABI) vs the reference's golden vectors and the CPU oracle."""
import numpy as np
import pytest

from risingwave_b200 import abi
from risingwave_b200.executor import HashJoinExecutor, JoinParams, MockSource
from risingwave_b200.stream_chunk import Column, StreamChunk, net_multiset, emitted_multiset

from helpers import JOIN_TYPES, load_golden, run_join_kat

pytestmark = pytest.mark.gpu

JOIN_KATS = [k for k in load_golden("hash_join_kats.json") if "skipped" not in k]


@pytest.mark.parametrize("kat", JOIN_KATS, ids=[k["name"] for k in JOIN_KATS])
def test_hash_join_golden(cuda, kat):
    """Every non-watermark test of hash_join.rs; order-insensitive (net applied multiset per step):
    the reference's own output order is not deterministic (SURVEY 0.2.8)."""
    run_join_kat(cuda, kat, exact=False)


def make_pair(cuda, oracle, jt, types, keys, pk, stream_key, null_safe, cond=None, append_only=False, chunk_size=1024):
    exs = []
    for be in (cuda, oracle):
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        exs.append(HashJoinExecutor(be, jt, sl.into_executor(types, stream_key), sr.into_executor(types, stream_key),
                                    JoinParams(keys, pk), JoinParams(keys, pk), null_safe, None, cond, append_only, chunk_size))
    return exs


class StreamGen:
    """Consistent two-sided change stream: deletes / updates always name a live row (unique pk per side)."""

    def __init__(self, seed, n_keys_cols=1, key_range=12, null_frac=0.0):
        self.rng = np.random.default_rng(seed)
        self.live = [[], []]
        self.next_pk = [0, 0]
        self.kc = n_keys_cols
        self.key_range = key_range
        self.null_frac = null_frac

    def new_row(self, side):
        r = self.rng
        keys = tuple(None if r.random() < self.null_frac else int(r.integers(0, self.key_range)) for _ in range(self.kc))
        pk = self.next_pk[side]
        self.next_pk[side] += 1
        payload = None if r.random() < self.null_frac else int(r.integers(0, 50))
        return keys + (pk, payload)

    def chunk(self, side, n, p_delete=0.25, p_update=0.15, types=None, vis_frac=1.0):
        rows = []
        r = self.rng
        live = self.live[side]
        while len(rows) < n:
            x = r.random()
            if live and x < p_delete:
                rows.append((abi.OP_DELETE, live.pop(int(r.integers(len(live)))), True))
            elif live and x < p_delete + p_update and len(rows) + 2 <= n:
                old = live.pop(int(r.integers(len(live))))
                new = old[:-1] + (int(r.integers(0, 50)),)  # same key & pk, new payload
                if r.random() < 0.3:  # key-changing update
                    new = tuple(int(r.integers(0, self.key_range)) for _ in range(self.kc)) + new[self.kc:]
                rows.append((abi.OP_UPDATE_DELETE, old, True))
                rows.append((abi.OP_UPDATE_INSERT, new, True))
                live.append(new)
            else:
                row = self.new_row(side)
                vis = r.random() < vis_frac
                rows.append((abi.OP_INSERT, row, vis))
                if vis:
                    live.append(row)
        ch = StreamChunk.from_rows(types, [(op, row) for op, row, _ in rows])
        vis = np.array([v for _, _, v in rows], dtype=bool)
        if not vis.all():
            ch.vis = vis
        return ch


def drive(exs, pushes):
    """pushes: list of (side, chunk). Compares the net applied multiset of every push."""
    total = 0
    for i, (side, ch) in enumerate(pushes):
        outs = [ex.eq_join_oneside(side, ch) for ex in exs]
        g, o = net_multiset(outs[0]), net_multiset(outs[1])
        assert g == o, f"push {i} side {side}: net output differs\n gpu-only {g - o}\n oracle-only {o - g}\ninput\n{ch}"
        for oc in outs[0]:
            assert oc.capacity() <= max(exs[0]._desc.chunk_size, 2) + 1
        total += sum(abs(v) for v in g.values())
    return total


ALL_TYPES = list(JOIN_TYPES.items())


@pytest.mark.parametrize("name,jt", ALL_TYPES, ids=[n for n, _ in ALL_TYPES])
def test_random_stream_all_join_types(cuda, oracle, name, jt):
    types = [abi.T_INT64, abi.T_INT64, abi.T_INT64]
    exs = make_pair(cuda, oracle, jt, types, [0], [1], [1], [False])
    gen = StreamGen(seed=10 + jt)
    pushes = []
    for i in range(24):
        side = int(gen.rng.integers(2))
        pushes.append((side, gen.chunk(side, int(gen.rng.integers(1, 200)), types=types)))
    drive(exs, pushes)


@pytest.mark.parametrize("name,jt", ALL_TYPES, ids=[n for n, _ in ALL_TYPES])
def test_random_stream_nulls_and_null_safe(cuda, oracle, name, jt):
    types = [abi.T_INT64, abi.T_INT32, abi.T_INT64, abi.T_INT64]
    exs = make_pair(cuda, oracle, jt, types, [0, 1], [2], [2], [True, False])
    gen = StreamGen(seed=40 + jt, n_keys_cols=2, key_range=4, null_frac=0.2)
    pushes = []
    for i in range(16):
        side = int(gen.rng.integers(2))
        pushes.append((side, gen.chunk(side, int(gen.rng.integers(1, 150)), types=types, vis_frac=0.9)))
    drive(exs, pushes)


@pytest.mark.parametrize("name", ["Inner", "LeftOuter", "FullOuter", "RightSemi", "LeftAnti"])
def test_random_stream_with_condition(cuda, oracle, name):
    types = [abi.T_INT64, abi.T_INT64, abi.T_INT64]
    exs = make_pair(cuda, oracle, JOIN_TYPES[name], types, [0], [1], [1], [False], cond="(less_than:boolean $2:int8 $5:int8)")
    gen = StreamGen(seed=77)
    pushes = []
    for i in range(16):
        side = int(gen.rng.integers(2))
        pushes.append((side, gen.chunk(side, int(gen.rng.integers(1, 150)), types=types)))
    drive(exs, pushes)


def test_same_pk_insert_delete_in_one_chunk(cuda, oracle):
    """`+ 3 8` then `- 3 8` in one chunk (hash_join.rs:1819-1823), U-/U+ with equal pk, and a
    delete-then-reinsert of the same pk: the sequential own-side rule."""
    types = [abi.T_INT64, abi.T_INT64]
    exs = make_pair(cuda, oracle, abi.JOIN_INNER, types, [0], [1], [1], [False])
    L, R = 0, 1
    pushes = [
        (L, StreamChunk.from_pretty(" I I\n + 3 8\n - 3 8\n + 3 9\n + 4 1")),
        (R, StreamChunk.from_pretty(" I I\n + 3 100\n + 4 101")),
        (L, StreamChunk.from_pretty(" I I\n - 3 9\n + 3 9\n - 3 9\n + 3 9\n U- 4 1\n U+ 4 1")),
        (R, StreamChunk.from_pretty(" I I\n + 3 102\n - 3 100")),
        (L, StreamChunk.from_pretty(" I I\n - 3 9\n - 4 1")),
        (R, StreamChunk.from_pretty(" I I\n + 3 103\n + 4 104")),
    ]
    drive(exs, pushes)


def test_strict_missing_delete(cuda):
    types = [abi.T_INT64, abi.T_INT64]
    for jt in (abi.JOIN_INNER, abi.JOIN_LEFT_OUTER):
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        ex = HashJoinExecutor(cuda, jt, sl.into_executor(types, [1]), sr.into_executor(types, [1]),
                              JoinParams([0], [1]), JoinParams([0], [1]), [False])
        with pytest.raises(abi.RwError) as e:
            ex.eq_join_oneside(0, StreamChunk.from_pretty(" I I\n - 1 1"))
        assert e.value.code == abi.RW_ERR_INCONSISTENT


def test_high_amplification_and_chunk_cut(cuda, oracle):
    """one key with 3000 build rows: a probe row emits 3000 rows cut into <= chunk_size chunks."""
    types = [abi.T_INT64, abi.T_INT64]
    exs = make_pair(cuda, oracle, abi.JOIN_INNER, types, [0], [1], [1], [False], chunk_size=256)
    n = 3000
    build = StreamChunk(np.full(n, abi.OP_INSERT, np.uint8), [Column(abi.T_INT64, np.full(n, 7, np.int64)), Column(abi.T_INT64, np.arange(n, dtype=np.int64))])
    probe = StreamChunk.from_pretty(" I I\n + 7 1\n + 8 2\n + 7 3")
    tot = drive(exs, [(1, build), (0, probe), (0, StreamChunk.from_pretty(" I I\n - 7 1"))])
    assert tot == 2 * n + n


def test_empty_and_ragged(cuda, oracle):
    types = [abi.T_INT64, abi.T_INT64]
    exs = make_pair(cuda, oracle, abi.JOIN_FULL_OUTER, types, [0], [1], [1], [False])
    gen = StreamGen(seed=5)
    pushes = [(0, StreamChunk.from_pretty(" I I")), (1, StreamChunk.from_pretty(" I I\n + 1 1 D"))]
    for n in (1, 63, 64, 65, 1025):
        pushes.append((n % 2, gen.chunk(n % 2, n, types=[abi.T_INT64] * 3).slice(0, n)))
    exs = make_pair(cuda, oracle, abi.JOIN_FULL_OUTER, [abi.T_INT64] * 3, [0], [1], [1], [False])
    drive(exs, [p for p in pushes if len(p[1].columns) == 3])


def test_large_inner_join_properties(cuda):
    """BASELINE cfg3 shape at reduced build size: 1M auctions (unique id) then 2M bids probing them.
    Size-independent properties: every bid matches exactly one auction (|out| == |bids|), the output
    preserves (bid payload, auction payload) pairing, and deleting all bids emits the exact inverse."""
    rng = np.random.default_rng(3)
    nb, npz = 1 << 20, 1 << 21
    ids = rng.permutation(nb).astype(np.int64)
    seller = rng.integers(0, 1000, nb).astype(np.int64)
    types = [abi.T_INT64, abi.T_INT64]
    _, sl = MockSource.channel()
    _, sr = MockSource.channel()
    ex = HashJoinExecutor(cuda, abi.JOIN_INNER, sl.into_executor(types, [1]), sr.into_executor(types, [0]),
                          JoinParams([0], [1]), JoinParams([0], []), [False], capacity_hint=nb)
    out = ex.eq_join_oneside(1, StreamChunk(np.full(nb, abi.OP_INSERT, np.uint8), [Column(abi.T_INT64, ids), Column(abi.T_INT64, seller)]))
    assert out == []
    auction = rng.integers(0, nb, npz).astype(np.int64)
    bidpk = np.arange(npz, dtype=np.int64)
    seller_of = np.zeros(nb, np.int64)
    seller_of[ids] = seller
    tot = 0
    chk = 0
    B = 1 << 18
    for i in range(0, npz, B):
        sl_ = slice(i, i + B)
        o = ex.eq_join_oneside(0, StreamChunk(np.full(B, abi.OP_INSERT, np.uint8), [Column(abi.T_INT64, auction[sl_]), Column(abi.T_INT64, bidpk[sl_])]))
        for c in o:
            assert (c.ops == abi.OP_INSERT).all() and c.vis is None
            a, b, rid, rs = (c.columns[k].data for k in range(4))
            assert np.array_equal(a, rid) and np.array_equal(rs, seller_of[a]) and np.array_equal(auction[b], a)
            tot += len(a)
            chk += int(b.sum())
    assert tot == npz and chk == int(bidpk.sum())
    # retract the first 2^18 bids: exact inverse
    o = ex.eq_join_oneside(0, StreamChunk(np.full(B, abi.OP_DELETE, np.uint8), [Column(abi.T_INT64, auction[:B]), Column(abi.T_INT64, bidpk[:B])]))
    assert sum(c.capacity() for c in o) == B and all((c.ops == abi.OP_DELETE).all() for c in o)
    # an auction update (U-/U+) now sees only the remaining bids
    cnt = np.bincount(auction[B:], minlength=nb)
    k = int(np.argmax(cnt))
    upd = StreamChunk.from_pretty(f" I I\n U- {k} {seller_of[k]}\n U+ {k} 5555")
    o = ex.eq_join_oneside(1, upd)
    # (cardinality: the extra-match area is reserved per warp in blocks of 64 rows, the unused part stays invisible)
    assert sum(c.cardinality() for c in o) == 2 * int(cnt[k])
    dels = sum(int(((c.ops == abi.OP_DELETE) & (c.vis if c.vis is not None else True)).sum()) for c in o)
    assert dels == int(cnt[k])


class StreamGen4(StreamGen):
    """StreamGen with a second payload column: rows are (key, pk, payload, payload2)."""

    def new_row(self, side):
        return super().new_row(side) + (int(self.rng.integers(0, 1 << 40)),)


def test_inner_key64_four_columns_large_chunks(cuda, oracle):
    """Inner join, one int64 key, 4 + 4 int64 columns = the quad-cooperative kernel (join_inner_q4_kernel):
    chunks large enough for many warps and overflow-pool refills, hot keys (several matches per row),
    deletes / updates, invisible rows, and the key that equals the table's EMPTY sentinel."""
    types = [abi.T_INT64] * 4
    exs = make_pair(cuda, oracle, abi.JOIN_INNER, types, [0], [1], [1], [False])
    gen = StreamGen4(seed=5, key_range=600)
    pushes = []
    for i in range(12):
        side = int(gen.rng.integers(2))
        pushes.append((side, gen.chunk(side, int(gen.rng.integers(300, 3000)), types=types, vis_frac=0.95)))
    total = drive(exs, pushes)
    assert total > 10000
    lo = -(1 << 63)
    sent = [(0, StreamChunk.from_rows(types, [(abi.OP_INSERT, (lo, 10 ** 9 + 1, 7, 8)), (abi.OP_INSERT, (lo, 10 ** 9 + 2, 9, 10))])),
            (1, StreamChunk.from_rows(types, [(abi.OP_INSERT, (lo, 10 ** 9 + 3, 1, 2)), (abi.OP_INSERT, (5, 10 ** 9 + 4, 3, 4))])),
            (0, StreamChunk.from_rows(types, [(abi.OP_DELETE, (lo, 10 ** 9 + 1, 7, 8))])),
            (1, StreamChunk.from_rows(types, [(abi.OP_UPDATE_DELETE, (lo, 10 ** 9 + 3, 1, 2)), (abi.OP_UPDATE_INSERT, (lo, 10 ** 9 + 3, 1, 99))]))]
    assert drive(exs, sent) > 0


def test_join_push_device_counted_matches_exact_chunk(cuda):
    """rwgpu_join_push_device_counted: a chunk whose buffers are larger than its row count, the count living
    on the device, gives the same output as the exact chunk (both through the quad-cooperative kernel)."""
    import torch
    from risingwave_b200 import device
    rng = np.random.default_rng(11)
    types = [abi.T_INT64] * 4
    nb, n, cap = 50000, 20000, 32768

    def make():
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        ex = HashJoinExecutor(cuda, abi.JOIN_INNER, sl.into_executor(types, [1]), sr.into_executor(types, [0]),
                              JoinParams([0], [1]), JoinParams([0], []), [False], capacity_hint=nb)
        ids = np.arange(nb, dtype=np.int64)
        cols = [torch.from_numpy(ids).cuda()] + [torch.from_numpy(rng.integers(0, 1000, nb).astype(np.int64)).cuda() for _ in range(3)]
        device.join_push_device(ex, abi.SIDE_RIGHT, device.DeviceChunk(torch.ones(nb, dtype=torch.uint8, device="cuda"), cols, types))
        return ex

    rng = np.random.default_rng(11)
    a = make()
    rng = np.random.default_rng(11)
    b = make()
    bid = [np.concatenate([rng.integers(0, nb + 100, n), np.full(cap - n, -77)]).astype(np.int64)] + \
          [np.concatenate([rng.integers(0, 1 << 30, n), np.full(cap - n, -1)]).astype(np.int64) for _ in range(3)]
    bid[1][:n] = np.arange(n)  # stream key
    ops = np.full(cap, abi.OP_INSERT, np.uint8)
    ops[rng.integers(0, n, 50)] = 0  # a few invisible rows
    full = [torch.from_numpy(c).cuda() for c in bid]
    ops_d = torch.from_numpy(ops).cuda()
    va = device.join_push_device(a, abi.SIDE_LEFT, device.DeviceChunk(ops_d[:n].contiguous(), [c[:n].contiguous() for c in full], types))
    got_a = (va.n_rows, va.ops().cpu().numpy(), [va.column(k).cpu().numpy() for k in range(va.n_cols)])
    count = torch.tensor([n], dtype=torch.int64, device="cuda")
    vb = device.join_push_device(b, abi.SIDE_LEFT, device.DeviceChunk(ops_d, full, types), n_rows_dev=count.data_ptr())
    got_b = (vb.n_rows, vb.ops().cpu().numpy(), [vb.column(k).cpu().numpy() for k in range(vb.n_cols)])
    assert got_a[0] == got_b[0] == n
    # positional output: row r of the output belongs to input row r; compare the visible rows
    def visible(view, got):
        import ctypes as C
        if view.vis_ptr is None:
            return np.ones(got[0], bool)
        words = torch.empty((got[0] + 63) // 64, dtype=torch.int64, device="cuda")
        device._d2d(words.data_ptr(), view.vis_ptr, words.numel() * 8)
        bits = np.unpackbits(words.cpu().numpy().view(np.uint8), bitorder="little")[:got[0]]
        return bits.astype(bool)
    ma, mb = visible(va, got_a), visible(vb, got_b)
    assert np.array_equal(ma, mb) and ma.sum() > n * 0.9
    assert np.array_equal(got_a[1][ma], got_b[1][mb])
    for ca, cb in zip(got_a[2], got_b[2]):
        assert np.array_equal(ca[ma], cb[mb])
    # a count outside [0, capacity] is rejected
    bad = torch.tensor([cap + 1], dtype=torch.int64, device="cuda")
    with pytest.raises(abi.RwError):
        device.join_push_device(b, abi.SIDE_LEFT, device.DeviceChunk(ops_d, full, types), n_rows_dev=bad.data_ptr())


# ------------------------------------------------------------------------------------------ unified-table path (round 2)
def _set_seq(cuda, ex, seq):
    import ctypes as C
    cuda.lib.rwgpu_join_debug_set_seq.restype = C.c_int32
    cuda.lib.rwgpu_join_debug_set_seq.argtypes = [C.c_void_p, C.c_uint64]
    assert cuda.lib.rwgpu_join_debug_set_seq(ex._h, C.c_uint64(seq)) == 0


@pytest.mark.parametrize("no_uni", [False, True], ids=["unified", "two_tables"])
@pytest.mark.parametrize("seq0", [(1 << 31) - 700, (1 << 32) - 700, (1 << 33) + 5], ids=["2^31", "2^32", "2^33"])
def test_delete_rule_across_arrival_counter_boundaries(cuda, oracle, monkeypatch, no_uni, seq0):
    """ADVICE r1 (high): the own-side delete picked its victim by a 32-bit wrap-aware age, so a live row inserted more
    than 2^31 arrivals ago could no longer be deleted.  Rows now carry a 64-bit arrival number; the counter is moved
    next to the boundaries through the test hook and a stream with deletes / same-pk re-inserts crosses them."""
    if no_uni:
        monkeypatch.setenv("RWGPU_NO_UNI", "1")
    types = [abi.T_INT64] * 4
    exs = make_pair(cuda, oracle, abi.JOIN_INNER, types, [0], [1], [1], [False])
    gen = StreamGen4(seed=21, key_range=40)
    # rows stored long BEFORE the boundary ...
    _set_seq(cuda, exs[0], 5)
    first = [(s, gen.chunk(s, 400, p_delete=0.0, p_update=0.0, types=types)) for s in (0, 1)]
    drive(exs, first)
    # ... are deleted / updated by chunks whose arrival numbers straddle it
    _set_seq(cuda, exs[0], seq0)
    pushes = []
    for i in range(10):
        side = i % 2
        pushes.append((side, gen.chunk(side, 300, p_delete=0.45, p_update=0.25, types=types)))
    pushes.append((0, StreamChunk.from_rows(types, [(abi.OP_INSERT, (3, 10 ** 9, 1, 2)), (abi.OP_DELETE, (3, 10 ** 9, 1, 2)),
                                                    (abi.OP_INSERT, (3, 10 ** 9, 1, 2)), (abi.OP_DELETE, (3, 10 ** 9, 1, 2)),
                                                    (abi.OP_INSERT, (3, 10 ** 9, 5, 6))])))
    pushes.append((1, StreamChunk.from_rows(types, [(abi.OP_INSERT, (3, 10 ** 9 + 1, 7, 8))])))
    assert drive(exs, pushes) > 1000


def test_unified_nulls_visibility_and_null_safe_key(cuda, oracle):
    """Key64 inner join with 4 + 4 columns (the unified-table path) fed chunks WITH validity / visibility bitmaps: NULL
    payload columns, NULL keys (never match, never stored) and, null-safe, NULL keys that do match each other."""
    types = [abi.T_INT64] * 4
    for null_safe in (False, True):
        exs = make_pair(cuda, oracle, abi.JOIN_INNER, types, [0], [1], [1], [null_safe])
        gen = StreamGen4(seed=33 + int(null_safe), key_range=25, null_frac=0.15)
        pushes = []
        for i in range(14):
            side = int(gen.rng.integers(2))
            pushes.append((side, gen.chunk(side, int(gen.rng.integers(50, 400)), types=types, vis_frac=0.9)))
        assert drive(exs, pushes) > 500


def test_unified_log_compaction_at_barrier(cuda, oracle):
    """An update-heavy stream: most stored rows die.  The barrier rebuilds a log that is more than half dead from its
    live records (the reference frees an entry at delete time, join/hash_join.rs:659-681); results stay identical."""
    types = [abi.T_INT64] * 4
    exs = make_pair(cuda, oracle, abi.JOIN_INNER, types, [0], [1], [1], [False])
    gen = StreamGen4(seed=77, key_range=500)
    total = 0
    for rnd in range(6):
        pushes = []
        for i in range(4):
            side = i % 2
            pushes.append((side, gen.chunk(side, 6000, p_delete=0.5 if rnd else 0.0, p_update=0.2 if rnd else 0.0, types=types)))
        total += drive(exs, pushes)
        for ex in exs:
            ex.flush_data(rnd + 1)
    assert total > 50000
    import ctypes as C
    cuda.lib.rwgpu_join_compactions.restype = C.c_uint64
    cuda.lib.rwgpu_join_compactions.argtypes = [C.c_void_p]
    assert cuda.lib.rwgpu_join_compactions(exs[0]._h) >= 1


def test_async_pushes_two_outstanding_match_synchronous(cuda):
    """rwgpu_join_push_device_async / rwgpu_join_collect: push s + 1 is launched before push s is collected (two output
    sets); every collected output equals the synchronous call's on an identical handle.  A push of the other side while
    one is outstanding is refused, so is a barrier."""
    import torch
    from risingwave_b200 import device
    rng = np.random.default_rng(5)
    types = [abi.T_INT64] * 4
    nb = 40000

    def make():
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        ex = HashJoinExecutor(cuda, abi.JOIN_INNER, sl.into_executor(types, [1]), sr.into_executor(types, [0]),
                              JoinParams([0], [1]), JoinParams([0], []), [False], capacity_hint=1000)  # small hint: growth on the way
        return ex

    auct = [np.arange(nb, dtype=np.int64)] + [rng.integers(0, 1000, nb).astype(np.int64) for _ in range(3)]
    bids = []
    for s in range(6):
        n = 30000 + 1000 * s
        cols = [rng.integers(0, nb + 50, n).astype(np.int64), (np.arange(n) + 10 ** 6 * s).astype(np.int64),
                rng.integers(0, 1 << 30, n).astype(np.int64), rng.integers(0, 1 << 30, n).astype(np.int64)]
        bids.append(cols)

    def dev(cols, ops=None):
        n = len(cols[0])
        o = torch.ones(n, dtype=torch.uint8, device="cuda") if ops is None else torch.from_numpy(ops).cuda()
        return device.DeviceChunk(o, [torch.from_numpy(c).cuda() for c in cols], types)

    def snapshot(v):
        vis = v.visible()
        cols = [v.column(k) for k in range(v.n_cols)]
        ops = v.ops()
        if vis is not None:
            cols, ops = [c[vis] for c in cols], ops[vis]
        return ops.cpu().numpy(), [c.cpu().numpy() for c in cols]

    a, b = make(), make()
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        for ex in (a, b):
            assert device.join_push_device(ex, abi.SIDE_RIGHT, dev(auct), stream).n_rows == 0
        want = [snapshot(device.join_push_device(a, abi.SIDE_LEFT, dev(c), stream)) for c in bids]
        chunks = [dev(c) for c in bids]
        got = []
        for s, ch in enumerate(chunks):
            device.join_push_device_async(b, abi.SIDE_LEFT, ch, stream)
            if s == 0:
                with pytest.raises(abi.RwError):  # other side while one is outstanding
                    device.join_push_device_async(b, abi.SIDE_RIGHT, dev(auct), stream)
                with pytest.raises(abi.RwError):
                    b.flush_data(1)
            if s > 0:
                got.append(snapshot(device.join_collect(b, stream)))
        got.append(snapshot(device.join_collect(b, stream)))
        with pytest.raises(abi.RwError):
            device.join_collect(b, stream)
    assert len(got) == len(want)
    for s, ((go, gc), (wo, wc)) in enumerate(zip(got, want)):
        assert np.array_equal(go, wo), f"push {s}"
        for x, y in zip(gc, wc):
            assert np.array_equal(x, y), f"push {s}"
    # the same protocol on a plan without an asynchronous kernel path (outer join): completes inside _async
    types2 = [abi.T_INT64] * 2
    _, sl = MockSource.channel()
    _, sr = MockSource.channel()
    ex = HashJoinExecutor(cuda, abi.JOIN_LEFT_OUTER, sl.into_executor(types2, [1]), sr.into_executor(types2, [1]),
                          JoinParams([0], [1]), JoinParams([0], [1]), [False])
    c2 = device.DeviceChunk(torch.ones(3, dtype=torch.uint8, device="cuda"),
                            [torch.tensor([1, 2, 3], device="cuda"), torch.tensor([7, 8, 9], device="cuda")], types2)
    device.join_push_device_async(ex, abi.SIDE_LEFT, c2)
    assert device.join_collect(ex).n_rows == 3


@pytest.mark.parametrize("shape", ["unified", "w8", "typed", "left_outer"])
def test_noop_update_pairs_are_hidden_like_the_reference(cuda, oracle, shape):
    """StreamChunk::eliminate_adjacent_noop_update (stream_chunk.rs:331-392, applied by JoinChunkBuilder::post_process): an
    update that does not change any OUTPUT column yields -x, +x on adjacent rows, and the reference hides both.  The
    device post-pass must hide exactly the same pairs: the multiset of rows actually EMITTED (visible) equals the
    oracle's, for streams where every row has at most one match (the row order of multi-match output is ours)."""
    if shape == "unified":
        types, out = [abi.T_INT64] * 3, [0, 1, 3, 4]          # payloads (cols 2, 5) projected away
    elif shape == "w8":
        types, out = [abi.T_INT64] * 6, [0, 1, 6, 7]
    elif shape == "typed":
        types, out = [abi.T_INT64, abi.T_INT32, abi.T_INT64], [0, 1, 3, 4]
    else:
        types, out = [abi.T_INT64] * 3, [0, 1, 3, 4]
    jt = abi.JOIN_LEFT_OUTER if shape == "left_outer" else abi.JOIN_INNER
    exs = []
    for be in (cuda, oracle):
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        exs.append(HashJoinExecutor(be, jt, sl.into_executor(types, [1]), sr.into_executor(types, [0]),
                                    JoinParams([0], [1]), JoinParams([0], [0]), [False], out, None, False, 64))  # small chunks: pairs straddle cuts
    rng = np.random.default_rng(3)
    nk = 300

    def row(k, pk, pay):
        return (k, pk, pay) + (7,) * (len(types) - 3)

    right = [(abi.OP_INSERT, row(k, k, int(rng.integers(0, 9)))) for k in range(nk)]
    left, pk = [], 0
    stored = {}
    perm = rng.permutation(nk)
    unused = [int(k) for k in perm[200:]]  # keys no left row uses: key-changing updates move here (every key keeps <= 1 left row)
    for k in perm[:200]:
        stored[pk] = (int(k), int(rng.integers(0, 9)))
        left.append((abi.OP_INSERT, row(int(k), pk, stored[pk][1])))
        pk += 1
    pushes = [(1, StreamChunk.from_rows(types, right)), (0, StreamChunk.from_rows(types, left))]
    # updates: half change only the payload (noop in the output), half change the key (a real change)
    upd = []
    for p_ in list(stored)[:150]:
        k, pay = stored[p_]
        nk2 = k
        if rng.random() < 0.5 and unused:
            nk2 = unused.pop()
            unused.insert(0, k)
        upd.append((abi.OP_UPDATE_DELETE, row(k, p_, pay)))
        upd.append((abi.OP_UPDATE_INSERT, row(nk2, p_, pay + 100)))
        stored[p_] = (nk2, pay + 100)
    pushes.append((0, StreamChunk.from_rows(types, upd)))
    # right-side payload updates: noop for every matching left row
    updr = []
    for k in range(0, nk, 2):
        r0 = right[k][1]
        updr.append((abi.OP_UPDATE_DELETE, r0))
        updr.append((abi.OP_UPDATE_INSERT, r0[:2] + (r0[2] + 50,) + r0[3:]))
    pushes.append((1, StreamChunk.from_rows(types, updr)))
    hidden = 0
    for i, (side, ch) in enumerate(pushes):
        g, o = (ex.eq_join_oneside(side, ch) for ex in exs)
        assert net_multiset(g) == net_multiset(o), f"push {i}"
        assert emitted_multiset(g) == emitted_multiset(o), f"push {i}: emitted rows differ"
        hidden += sum(int((~c.vis).sum()) for c in g if c.vis is not None)
    assert hidden > 0


# ------------------------------------------------------------------------------------------ varlen payload columns (round 2)
@pytest.mark.parametrize("name", ["Inner", "LeftOuter", "RightSemi"])
def test_varlen_payload_columns_travel_through_the_join(cuda, oracle, name):
    """varchar columns (BytesArray{offset, bitmap, data}, bytes_array.rs:30-34) as PAYLOAD: interned into the side's byte
    heap on the way in, gathered back into offsets + bytes on the way out; NULL and empty strings, deletes, updates that
    change only the string, snapshot / restore -- vs the oracle."""
    jt = JOIN_TYPES[name]
    tl = [abi.T_INT64, abi.T_INT64, abi.T_VARCHAR, abi.T_INT64]      # bid-like: auction, row id, url, price
    tr = [abi.T_INT64, abi.T_VARCHAR, abi.T_VARCHAR]                 # auction-like: id, item name, description
    rng = np.random.default_rng(23)
    words = [b"", b"a", b"url-" + bytes(range(65, 91)), b"\xf0\x9f\x9a\x80 unicode", b"x" * 300, None]

    def mk(be):
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        return HashJoinExecutor(be, jt, sl.into_executor(tl, [1]), sr.into_executor(tr, [0]), JoinParams([0], [1]), JoinParams([0], [0]), [False])

    g, o = mk(cuda), mk(oracle)
    live = [dict(), dict()]
    next_pk = [0]

    def w():
        return words[int(rng.integers(len(words)))]

    def chunk(side, n):
        rows = []
        while len(rows) < n:
            x = rng.random()
            lv = live[side]
            if lv and x < 0.2:
                k = list(lv)[int(rng.integers(len(lv)))]
                rows.append((abi.OP_DELETE, lv.pop(k)))
            elif lv and x < 0.35 and len(rows) + 2 <= n:
                k = list(lv)[int(rng.integers(len(lv)))]
                old = lv[k]
                new = (old[:2] + (w(),) + old[3:]) if side == 0 else (old[:1] + (w(),) + old[2:])
                rows += [(abi.OP_UPDATE_DELETE, old), (abi.OP_UPDATE_INSERT, new)]
                lv[k] = new
            elif side == 0:
                next_pk[0] += 1
                row = (int(rng.integers(0, 60)), next_pk[0], w(), int(rng.integers(0, 1000)))
                rows.append((abi.OP_INSERT, row))
                lv[row[1]] = row
            else:
                k = int(rng.integers(0, 60))
                if k in lv:
                    continue
                row = (k, w(), w())
                rows.append((abi.OP_INSERT, row))
                lv[k] = row
        return StreamChunk.from_rows(tl if side == 0 else tr, rows)

    for i in range(14):
        side = int(rng.integers(2))
        ch = chunk(side, int(rng.integers(20, 400)))
        assert net_multiset(g.eq_join_oneside(side, ch)) == net_multiset(o.eq_join_oneside(side, ch)), f"push {i}"
    # state persistence with varlen columns
    snaps = [g.snapshot(s) for s in (0, 1)]
    for s in (0, 1):
        assert sorted((r for c in snaps[s] for _, r in c.rows()), key=repr) == sorted(live[s].values(), key=repr)
    g2 = mk(cuda)
    for s in (0, 1):
        if snaps[s]:
            from risingwave_b200.stream_chunk import concat_chunks
            g2.restore(s, concat_chunks(snaps[s]))
    for i in range(6):
        side = int(rng.integers(2))
        ch = chunk(side, int(rng.integers(20, 300)))
        want = net_multiset(o.eq_join_oneside(side, ch))
        assert net_multiset(g.eq_join_oneside(side, ch)) == want, f"after snapshot, push {i}"
        assert net_multiset(g2.eq_join_oneside(side, ch)) == want, f"restored operator, push {i}"


def test_varlen_key_or_pk_is_refused(cuda):
    for types, keys, pk in (([abi.T_VARCHAR, abi.T_INT64], [0], [1]), ([abi.T_INT64, abi.T_VARCHAR], [0], [1])):
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        with pytest.raises(abi.RwError) as e:
            HashJoinExecutor(cuda, abi.JOIN_INNER, sl.into_executor(types, [1]), sr.into_executor(types, [1]), JoinParams(keys, pk), JoinParams(keys, pk),
                             [False])
        assert e.value.code == abi.RW_ERR_UNSUPPORTED


def test_host_async_pushes_match_synchronous(cuda, oracle):
    """rwgpu_join_push_async / rwgpu_join_collect_out (host chunks, two outstanding): every collected output equals the
    synchronous rwgpu_join_push on an identical handle and the oracle's net result -- inserts with 0 / 1 / many matches
    (extra rows copied at collect), deletes (ops re-copied after the no-op pass), NULL payload (validity bytes), invisible
    input rows, and an amplification above the 2x host block (re-laid at collect)."""
    rng = np.random.default_rng(77)
    types = [abi.T_INT64] * 4
    nb = 5000

    def make(be):
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        return HashJoinExecutor(be, abi.JOIN_INNER, sl.into_executor(types, [1]), sr.into_executor(types, [0]),
                                JoinParams([0], [1]), JoinParams([0], []), [False], capacity_hint=1000)

    a, b, o = make(cuda), make(cuda), make(oracle)
    auct_cols = [np.arange(nb, dtype=np.int64)] + [rng.integers(0, 1000, nb).astype(np.int64) for _ in range(3)]
    valid3 = rng.random(nb) > 0.1
    auct = StreamChunk(np.full(nb, abi.OP_INSERT, np.uint8), [Column(abi.T_INT64, c) for c in auct_cols[:3]] + [Column(abi.T_INT64, auct_cols[3], valid3)])
    for ex in (a, b, o):
        assert ex.eq_join_oneside(1, auct) == []
    pushes = []
    stored = []
    for s in range(7):
        n = 20000 + 3000 * s
        key = rng.integers(0, nb + 500, n).astype(np.int64)  # some bids match nothing
        pk = (np.arange(n) + 10 ** 6 * s).astype(np.int64)
        cols = [key, pk, rng.integers(0, 1 << 30, n).astype(np.int64), rng.integers(0, 1 << 30, n).astype(np.int64)]
        ops = np.full(n, abi.OP_INSERT, np.uint8)
        vis = None
        if s == 3:  # retract rows of an earlier push
            k0, p0, c2, c3 = stored[0]
            cols = [k0[:5000], p0[:5000], c2[:5000], c3[:5000]]
            ops = np.full(5000, abi.OP_DELETE, np.uint8)
        elif s == 4:
            vis = rng.random(n) > 0.2
        else:
            stored.append(cols)
        pushes.append((0, StreamChunk(ops, [Column(abi.T_INT64, c) for c in cols], vis)))
    # auction updates: every bid of the auction is emitted twice (extra-match rows; > 2x the input for the hot ones).  The
    # update changes a column that is never NULL: with an unchanged output row the no-op pass would hide whichever pair of
    # matches lands adjacent, and the order of a key's matches is not part of the result
    hot = np.repeat(np.arange(40, dtype=np.int64), 2)
    upd_ops = np.tile(np.array([abi.OP_UPDATE_DELETE, abi.OP_UPDATE_INSERT], np.uint8), 40)
    upd_cols = [hot] + [np.repeat(c[:40], 2) for c in auct_cols[1:]]
    upd_cols[2] = upd_cols[2] + np.tile(np.array([0, 1], np.int64), 40)
    hot_bids = StreamChunk(np.full(4000, abi.OP_INSERT, np.uint8),
                           [Column(abi.T_INT64, rng.integers(0, 40, 4000).astype(np.int64)), Column(abi.T_INT64, np.arange(4000, dtype=np.int64) + 10 ** 9),
                            Column(abi.T_INT64, np.zeros(4000, np.int64)), Column(abi.T_INT64, np.ones(4000, np.int64))])
    pushes.append((0, hot_bids))
    pushes.append((1, StreamChunk(upd_ops, [Column(abi.T_INT64, c) for c in upd_cols[:3]] + [Column(abi.T_INT64, upd_cols[3], np.repeat(valid3[:40], 2))])))

    def rows_of(chunks):
        return sorted((int(op), tuple(None if v is None else int(v) for v in row)) for ch in chunks for op, row in ch.rows())

    want = [rows_of(a.eq_join_oneside(side, ch)) for side, ch in pushes]
    want_net = [net_multiset(o.eq_join_oneside(side, ch)) for side, ch in pushes]
    got = []
    outstanding = []
    for side, ch in pushes:
        if outstanding and outstanding[-1] != side:  # pushes of different sides are never outstanding together
            while outstanding:
                got.append(rows_of(b.eq_join_oneside_collect()))
                outstanding.pop(0)
        b.eq_join_oneside_launch(side, ch)
        outstanding.append(side)
        if len(outstanding) == 2:
            got.append(rows_of(b.eq_join_oneside_collect()))
            outstanding.pop(0)
    while outstanding:
        got.append(rows_of(b.eq_join_oneside_collect()))
        outstanding.pop(0)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, f"push {i}"
    from collections import Counter
    for i, g in enumerate(got):
        net = Counter()
        for op, row in g:
            net[row] += 1 if op in (abi.OP_INSERT, abi.OP_UPDATE_INSERT) else -1
        assert {k: v for k, v in net.items() if v} == {k: v for k, v in dict(want_net[i]).items() if v}, f"push {i} vs oracle"
    # a third launch without a collect is refused; so is a device collect of a host launch
    b.eq_join_oneside_launch(0, pushes[0][1])
    b.eq_join_oneside_launch(0, pushes[1][1])
    with pytest.raises(abi.RwError):
        b.eq_join_oneside_launch(0, pushes[2][1])
    b.eq_join_oneside_collect()
    b.eq_join_oneside_collect()
