"""-m gpu: the device ingest for every fold program and engine path, against the host ingest and an independent oracle.

tests/test_gpu_dingest.py folds the Counter program with default options only, so every poll there takes the sort-free atomic
fold, which skips the holes the device decode leaves in place of dropped records (flush markers, duplicates, null values: an
aggregate index of UINT64_MAX). Any other program, any non-default option and the deferred throw replay take the sort-based
path (stable group-by + fold). Here the same wire bytes go through
  1. the device ingest (DeviceIngest + the engine),
  2. the host decoder (Ingest + ReplayEngine.fold_ingested),
  3. a reference chain that shares no code with either: oracle.kafka_batch.read_committed_pack (wire -> packed records, first-seen
     ids, next offsets) -> oracle.program_interp.fold_arrival_order, one fold per poll onto a live table; the C oracle
     (oracle.oracle.fold_incremental, the sample models' handlers) where the interpreter would be too slow,
and every poll must agree per id on program bytes, flags and err_idx, on partition offsets and on the poll's statistics. Device
slots no id maps to must stay all-zero: a hole folded into some slot shows up there.

Also here: the engine-level hole contract of every arrival-order entry point, and the replay-list overflow of the record-parallel
fold (full fold: sequential redo; in-place incremental fold: table invalidated until the caller resets it).
"""
import struct

import numpy as np
import pytest

from oracle import kafka_batch as K
from oracle import oracle as O
from oracle import program_interp as I
from surge_b200 import ReplayEngine, SgrError
from surge_b200 import native as N
from surge_b200.native import InvalidStateStoreException
from surge_b200 import programs as P
from surge_b200.dingest import DeviceIngest
from surge_b200.ingest import Ingest, IngestError
from test_gpu_program_fuzz import SPECIAL_F64, draw_program, same

pytestmark = pytest.mark.gpu

HOLE = (1 << 64) - 1
POLL_STATS = ("n_records", "n_markers", "n_null_values", "n_duplicates", "n_new_keys")
REDO_CAP = 1 << 20          # throwing aggregates the record-parallel kernel's replay list holds (engine.cu kRedoCap)


def _rules_of(prog):
    return [(int(prog.rules[t].exists_rule), [(int(o.opcode), int(o.dst_off), int(o.src_off), int(o.len)) for o in prog.rules[t].ops[:prog.rules[t].n_ops]])
            for t in range(prog.n_types)]


# ------------------------------------------------------------------ programs and the event values they read
class Program:
    def __init__(self, name, prog, value, null_type=None):
        self.name, self.prog, self.value, self.null_type = name, prog, value, null_type
        self.rules = _rules_of(prog)
        self.state_bytes = int(prog.state_bytes)
        self.f64 = [int(prog.f64_field_off[i]) for i in range(prog.n_f64_fields)]
        # record bytes 8..16 hold the aggregate index, which the device ingest assigns in another order than the host
        assert all(src >= 16 or src + ln <= 8 for _, ops in self.rules for _, _, src, ln in ops), name


def _counter_value(types, p):
    def value(rng, seq):
        t = int(rng.choice(types, p=p))
        return struct.pack("<IIi", t, seq, int(rng.integers(-2**31, 2**31))) + rng.bytes(int(rng.integers(0, 37)))
    return value


def _bank_value(rng, seq):
    """BankAccount events: 56-byte values (uuid, balance, owner, code); type 2 is a MatchError. Balances include +-0.0 and NaN,
    which the publish rule compares with JVM == (CHANGED or not)."""
    t = int(rng.choice([0, 1, 2], p=[0.3, 0.62, 0.08]))
    bal = float(SPECIAL_F64[int(rng.integers(0, len(SPECIAL_F64)))]) if rng.random() < 0.6 else float(rng.integers(-5, 5))
    return struct.pack("<II", t, seq) + rng.bytes(16) + struct.pack("<d", bal) + rng.bytes(24)


def _random_value(n_types, f64):
    def value(rng, seq):
        t = n_types if rng.random() < 0.03 else int(rng.integers(0, n_types))   # type >= n_types: scala.MatchError
        payload = bytearray(rng.bytes(48))
        if f64 and rng.random() < 0.5:
            payload[16:24] = struct.pack("<d", SPECIAL_F64[int(rng.integers(0, len(SPECIAL_F64)))])   # record bytes 24..32
        return struct.pack("<II", t, seq) + bytes(payload[:int(rng.integers(0, 49))])
    return value


def _programs():
    out = [
        Program("counter", P.counter_program(), _counter_value([0, 1, 2, 3], [0.45, 0.3, 0.15, 0.1])),
        Program("counter_snapshot", P.counter_program_with_snapshot_rules(), _counter_value([0, 1, 2, 3, 4, 5], [0.3, 0.2, 0.1, 0.05, 0.3, 0.05]),
                null_type=P.COUNTER_TOMBSTONE_TYPE),
        Program("ml_counter", P.ml_counter_program(), _counter_value([0, 1, 2, 3], [0.5, 0.35, 0.1, 0.05])),
        Program("int_balance", P.int_balance_program(), _counter_value([0, 1], [0.93, 0.07])),
        Program("bank_account", P.bank_account_program(), _bank_value),
    ]
    seed = 4400
    while len(out) < 13:
        sb, rules, f64 = draw_program(np.random.default_rng(seed))
        seed += 1
        if any(ex in (I.MATERIALISE, I.CREATE) for ex, _ in rules):     # a program that never creates a state checks little
            out.append(Program(f"random{seed - 1}", P.make_program(sb, N.REC_FIXED64, rules, f64_fields=f64), _random_value(len(rules), f64)))
    return out


PROGRAMS = _programs()
OPTIONS = {"default": {}, "incremental1": {"incremental": 1}, "kernel1": {"kernel": 1}, "replay_budget0": {"replay_budget": 0}}


# ------------------------------------------------------------------ polls
def _draw_polls(rng, prog, n_polls=3):
    """Polls of three partitions. Every poll has flush markers (empty key), null values, new ids, throwing events; partition 0
    re-sends its previous last batch (a refetch below the folded position: duplicates), partition 1 has an aborted and a
    committed transaction. Returns [[(partition, wire, aborted, oracle_wire)]]: oracle_wire is the same batches with each null
    value written as the event the state-topic mode makes of it, `u32 null_type, u32 seq = 0` and zeros (read_committed_pack
    drops null values, which is what the product does without a null-value type)."""
    nxt = {0: 0, 1: 0, 2: 0}
    last0 = (b"", b"")
    polls = []
    for k in range(n_polls):
        poll = []
        n_ids = 20 * (k + 1)
        for part in range(3):
            wire, owire, aborted = bytearray(), bytearray(), []
            if part == 0 and k:
                wire += last0[0]; owire += last0[1]
            for j in range(int(rng.integers(2, 5))):
                off = nxt[part]
                recs, orecs = [], []
                for d in range(int(rng.integers(1, 14))):
                    u = rng.random()
                    key = f"agg-{int(rng.integers(0, n_ids))}".encode() + (b":%d" % (off + d) if rng.random() < 0.5 else b"")
                    if u < 0.07:
                        recs.append((d, b"", b"")); orecs.append((d, b"", b""))
                    elif u < 0.14:
                        recs.append((d, key, None))
                        orecs.append((d, key, None if prog.null_type is None else struct.pack("<II", prog.null_type, 0)))
                    else:
                        v = prog.value(rng, off + d + 1)
                        recs.append((d, key, v)); orecs.append((d, key, v))
                comp = "lz4" if rng.random() < 0.4 else "none"
                kind = "aborted" if (part, j) == (1, 0) else "committed" if (part, j) == (1, 1) else "plain"
                if kind == "plain":
                    b, ob = K.encode_record_batch(off, recs, compression=comp), K.encode_record_batch(off, orecs, compression=comp)
                    nxt[part] = off + len(recs)
                    if part == 0:
                        last0 = (b, ob)
                else:
                    pid = 1000 + 10 * k + j
                    b = K.encode_record_batch(off, recs, compression=comp, producer_id=pid, transactional=True)
                    ob = K.encode_record_batch(off, orecs, compression=comp, producer_id=pid, transactional=True)
                    ctl = K.encode_control_batch(off + len(recs), pid, K.ABORT if kind == "aborted" else K.COMMIT)
                    b, ob = b + ctl, ob + ctl
                    if kind == "aborted":
                        aborted.append((pid, off))
                    nxt[part] = off + len(recs) + 1
                wire += b; owire += ob
            poll.append((part, bytes(wire), aborted, bytes(owire)))
        polls.append(poll)
    return polls


def _check_tables(what, ed, eh, ing, keys, table):
    """Host table rows are first-seen ids; device rows come from the device's own index of each id. Unmapped slots: all zero."""
    assert ing.keys() == keys, what
    host = eh.export_states()
    same(host[:len(keys)], table, f"{what}: host ingest")
    assert not host[len(keys):].any(), f"{what}: host slots without an id are not empty"
    dev = ed.export_states()
    idx = [ed.index_of(k) for k in keys]
    assert None not in idx, f"{what}: ids missing from the device key table: {[k for k, i in zip(keys, idx) if i is None][:5]}"
    idx = np.asarray(idx, dtype=np.int64)
    assert len(np.unique(idx)) == len(keys), f"{what}: two ids share a device slot"
    same(dev[idx], table, f"{what}: device ingest (rows in oracle id order)")
    unmapped = np.ones(len(dev), dtype=bool)
    unmapped[idx] = False
    dirty = np.nonzero(unmapped & dev.any(axis=1))[0]
    assert not len(dirty), f"{what}: device slots no id maps to were written: {dirty[:6]} {dev[dirty[0]].tolist()}"
    for k in keys[::7]:                                   # sgr_get resolves the same index
        want = table[keys.index(k)]
        flags = int(want[-8:-4].view(np.uint32)[0])
        assert ed.get(k) == (want[:-8].tobytes() if flags & N.ST_EXISTS else None), f"{what}: get({k})"


@pytest.mark.parametrize("option", list(OPTIONS))
@pytest.mark.parametrize("prog", PROGRAMS, ids=[p.name for p in PROGRAMS])
def test_device_ingest_matches_host_and_oracle(prog, option):
    rng = np.random.default_rng(77 + PROGRAMS.index(prog))
    polls = _draw_polls(rng, prog)
    sb = prog.state_bytes
    with ReplayEngine(0) as ed, ReplayEngine(0) as eh:
        for e in (ed, eh):
            e.register_program(prog.prog)
            for name, v in OPTIONS[option].items():
                e.set_option(name, v)
        ing = Ingest()
        with DeviceIngest(ed, 1 << 12) as dg:
            if prog.null_type is not None:
                dg.set_null_value_type(prog.null_type)
                ing.set_null_value_type(prog.null_type)
            fetches, n_prev = [], 0
            table = np.zeros((0, sb), dtype=np.uint8)
            for k, poll in enumerate(polls):
                what = f"{prog.name} {option} poll {k}"
                host_st = dict.fromkeys(POLL_STATS, 0)
                for part, wire, aborted, owire in poll:
                    dg.set_aborted(part, aborted)
                    ing.set_aborted(part, aborted)
                    dg.submit(part, wire)
                    hs = ing.record_batches(part, wire)
                    for s in POLL_STATS:
                        host_st[s] += hs[s]
                    fetches.append((part, owire, aborted))
                st = dg.fold()
                eh.fold_ingested(ing)
                recs, keys, nxt = K.read_committed_pack(fetches)
                keys = [k.decode() for k in keys]
                batch, n_prev = recs[n_prev:], len(recs)
                table = np.vstack([table, np.zeros((len(keys) - len(table), sb), dtype=np.uint8)])
                table = I.fold_arrival_order(prog.rules, sb, batch, table, f64_fields=prog.f64)
                assert {s: st[s] for s in POLL_STATS} == host_st, what
                assert host_st["n_records"] == len(batch), what
                for part in nxt:
                    assert dg.offsets(part) == ing.offsets(part) == (nxt[part], nxt[part]), f"{what} partition {part}"
                _check_tables(what, ed, eh, ing, keys, table)
            tot = ing.stats()
            assert min(tot["n_markers"], tot["n_null_values"], tot["n_duplicates"], tot["n_aborted_records"]) > 0, tot


def test_failed_fold_keeps_the_key_table_in_step():
    """A poll whose fold fails after its new ids reached the engine's key table (here: a 64-byte program with the record-per-lane
    kernel forced, which refuses it) is fetched again and followed by a poll with more new ids. Every id must still resolve to
    its own slot: appending the failed poll's ids a second time would shift every later id onto another aggregate's state."""
    prog = next(p for p in PROGRAMS if p.name == "bank_account")
    rng = np.random.default_rng(5)

    def clean_batch(off, ids):
        return K.encode_record_batch(off, [(d, b"acct-%d" % i, prog.value(rng, off + d + 1)) for d, i in enumerate(ids)])

    p1 = clean_batch(0, range(40))
    p2 = clean_batch(40, list(range(30, 70)) + list(range(70, 90)))
    p3 = clean_batch(100, list(range(85, 130)))
    sb = prog.state_bytes
    with ReplayEngine(0) as ed:
        ed.register_program(prog.prog)
        with DeviceIngest(ed, 1 << 12) as dg:
            dg.submit(0, p1)
            dg.fold()
            ed.set_option("kernel", 3)
            dg.submit(0, p2)
            with pytest.raises(IngestError) as ei:
                dg.fold()
            assert ei.value.code == N.SGR_ERR_UNSUPPORTED, ei.value
            assert dg.offsets(0) == (40, 40)
            ed.set_option("kernel", 0)
            dg.submit(0, p2)                                  # fetched again from the folded position
            dg.submit(0, p3)
            st = dg.fold()
            assert st["n_new_keys"] == 90, st
            recs, keys, _ = K.read_committed_pack([(0, p1, []), (0, p2, []), (0, p3, [])])
            keys = [k.decode() for k in keys]
            n1 = 40
            table = I.fold_arrival_order(prog.rules, sb, recs[:n1], np.zeros((n1, sb), dtype=np.uint8), f64_fields=prog.f64)
            table = np.vstack([table, np.zeros((len(keys) - n1, sb), dtype=np.uint8)])
            table = I.fold_arrival_order(prog.rules, sb, recs[n1:], table, f64_fields=prog.f64)
            dev = ed.export_states()
            for j, k in enumerate(keys):
                i = ed.index_of(k)
                assert i is not None and i < len(dev), (k, i)
                same(dev[i:i + 1], table[j:j + 1], f"id {k} -> slot {i}")
                flags = int(table[j, -8:-4].view(np.uint32)[0])
                assert ed.get(k) == (table[j, :-8].tobytes() if flags & N.ST_EXISTS else None), k


def _counter_records(agg, types, seqs, bys):
    r = np.zeros((len(agg), 64), dtype=np.uint8)
    r[:, 0:4] = np.asarray(types, dtype="<u4").view(np.uint8).reshape(-1, 4)
    r[:, 4:8] = np.asarray(seqs, dtype="<u4").view(np.uint8).reshape(-1, 4)
    r[:, 8:16] = np.asarray(agg, dtype="<u8").view(np.uint8).reshape(-1, 8)
    r[:, 16:20] = np.asarray(bys, dtype="<i4").view(np.uint8).reshape(-1, 4)
    return r


def test_replay_at_a_table_of_exactly_65536_slots():
    """65 536 ids make the device table exactly 2^16 slots, so a hole's index (UINT64_MAX) and slot 65 535 share every digit of
    a 16-bit radix sort. Poll 2 throws on every id after holes (markers, null values, a refetch) and, with replay_budget=0, every
    throwing slot goes through the deferred replay's group-by. The whole table must equal the oracle."""
    n = 1 << 16
    rng = np.random.default_rng(65536)
    ids = np.arange(n, dtype=np.uint32)
    t1 = np.zeros(n, dtype=np.uint32)
    s1 = np.arange(1, n + 1, dtype=np.uint32)
    b1 = rng.integers(-1000, 1000, size=n).astype(np.int32)
    head = n - 512
    w1a = O.kafka_encode_counter(ids[:head], t1[:head], s1[:head], b1[:head], recs_per_batch=512, lz4=False).tobytes()
    w1b = O.kafka_encode_counter(ids[head:], t1[head:], s1[head:], b1[head:], recs_per_batch=512, lz4=False, base_offset=head).tobytes()
    # poll 2: the refetched last batch, then per id an increment and later a throw, and some events after the throws (dropped);
    # a batch of flush markers and null values after every 4096 records
    order_inc, order_thr, order_after = rng.permutation(n), rng.permutation(n), rng.permutation(n)[:5000]
    agg2 = np.concatenate([order_inc, order_thr, order_after]).astype(np.uint32)
    typ2 = np.concatenate([np.zeros(n), np.full(n, 3), rng.integers(0, 3, size=len(order_after))]).astype(np.uint32)
    seq2 = np.arange(len(agg2), dtype=np.uint32) + n + 1
    by2 = rng.integers(-1000, 1000, size=len(agg2)).astype(np.int32)
    wire2, off = bytearray(w1b), n
    for c in range(0, len(agg2), 4096):
        sl = slice(c, c + 4096)
        cnt = len(agg2[sl])
        wire2 += O.kafka_encode_counter(agg2[sl], typ2[sl], seq2[sl], by2[sl], recs_per_batch=512, lz4=False, base_offset=off).tobytes()
        off += cnt
        junk = [(0, b"", b""), (1, b"agg-%d" % int(rng.integers(0, n)), None), (2, b"", b"")]
        wire2 += K.encode_record_batch(off, junk)
        off += len(junk)
    want = O.fold_incremental(O.MODEL_COUNTER, _counter_records(ids, t1, s1, b1), np.zeros((n, 16), dtype=np.uint8))
    want = O.fold_incremental(O.MODEL_COUNTER, _counter_records(agg2, typ2, seq2, by2), want)
    keys = [f"agg-{i}" for i in range(n)]
    with ReplayEngine(0) as ed, ReplayEngine(0) as eh:
        ing = Ingest()
        for e in (ed, eh):
            e.register_program(P.counter_program())
            e.set_option("replay_budget", 0)
        with DeviceIngest(ed, 1 << 17) as dg:
            dg.submit(0, w1a + w1b)
            dg.fold()
            assert ed.n_aggregates() == n
            dg.submit(0, bytes(wire2))
            st = dg.fold()
            assert st["n_duplicates"] == 512 and st["n_markers"] > 0 and st["n_null_values"] > 0 and st["n_new_keys"] == 0, st
            assert ed.n_aggregates() == n
            ing.record_batches(0, w1a + w1b)
            eh.fold_ingested(ing)
            ing.record_batches(0, bytes(wire2))
            eh.fold_ingested(ing)
            same(eh.export_states()[:n], want, "host ingest")
            idx = np.asarray([ed.index_of(k) for k in keys], dtype=np.int64)
            assert sorted(idx.tolist()) == list(range(n))
            dev = ed.export_states()
            last = keys[int(np.nonzero(idx == n - 1)[0][0])]
            same(dev[idx], want, f"device ingest (slot {n - 1} is {last})")
            assert ed.stats().n_errors == n


# ------------------------------------------------------------------ B. the engine-level hole contract
def _draw_batch(rng, n_types, n_agg, n):
    rec = rng.integers(0, 256, size=(n, 64), dtype=np.uint8)
    types = rng.integers(0, n_types, size=n).astype(np.uint32)
    types[rng.random(n) < 0.02] = n_types                     # scala.MatchError
    rec[:, 0:4] = types.view(np.uint8).reshape(-1, 4)
    rec[:, 4:8] = np.arange(1, n + 1, dtype=np.uint32).view(np.uint8).reshape(-1, 4)
    agg = rng.integers(0, n_agg, size=n).astype(np.uint64)
    agg[rng.integers(0, n, size=8)] = n_agg - 1               # the last slot, which a hole aliases in a too-narrow sort
    rec[:, 8:16] = agg.view(np.uint8).reshape(-1, 8)
    return rec


def _with_holes(rng, rec, n_holes):
    holes = rng.integers(0, 256, size=(n_holes, 64), dtype=np.uint8)   # whatever a dropped record leaves: never read
    holes[:, 8:16] = np.full(n_holes, HOLE, dtype=np.uint64).view(np.uint8).reshape(-1, 8)
    at = np.sort(rng.integers(0, len(rec) + 1, size=n_holes))
    return np.insert(rec, at, holes, axis=0)


HOLE_PATHS = {"atomic": {}, "sorted": {"incremental": 1}, "replay": {"replay_budget": 0}}


def _hole_programs(rng):
    out = [(16, _rules_of(P.counter_program()), [])]
    for _ in range(2):
        out.append(draw_program(rng))
    return out


def _stats_tuple(e):
    s = e.stats()
    return s.n_events, s.n_errors, s.n_aggregates


@pytest.mark.parametrize("n_agg", [256, 1000, 65536])
@pytest.mark.parametrize("path", list(HOLE_PATHS))
def test_holes_are_skipped_by_every_arrival_order_entry_point(path, n_agg):
    """agg == UINT64_MAX is a hole (include/sgr.h): fold_incremental, fold_unsorted and load_unsorted give exactly what the same
    batch without its holes gives, states and statistics; any other index >= n_agg is SGR_ERR_INVALID with nothing applied."""
    rng = np.random.default_rng(n_agg * 7 + len(path))
    for sb, rules, f64 in _hole_programs(rng):
        prog = P.make_program(sb, N.REC_FIXED64, rules, f64_fields=f64)
        what = f"{path} n_agg {n_agg} state_bytes {sb} rules {rules}"
        base = _draw_batch(rng, len(rules), n_agg, 3 * n_agg)
        batch = _draw_batch(rng, len(rules), n_agg, max(n_agg // 2, 300))
        holey = _with_holes(rng, batch, max(len(batch) // 10, 5))
        with ReplayEngine(0) as e:
            e.register_program(prog)
            for name, v in HOLE_PATHS[path].items():
                e.set_option(name, v)
            got = {}
            for label, recs in (("clean", batch), ("holes", holey)):
                e.set_initial_states(None)
                e.fold_unsorted(base, n_agg)
                e.fold_incremental(recs)
                inc = (e.export_states(), _stats_tuple(e))
                e.set_initial_states(None)
                e.fold_unsorted(recs, n_agg)
                unsorted = (e.export_states(), _stats_tuple(e))
                e.set_initial_states(None)
                e.load_unsorted(recs, n_agg)
                e.fold()
                loaded = (e.export_states(), _stats_tuple(e))
                got[label] = (inc, unsorted, loaded)
            for name, c, h in zip(("fold_incremental", "fold_unsorted", "load_unsorted"), got["clean"], got["holes"]):
                same(h[0], c[0], f"{what}: {name} with holes")
                assert h[1] == c[1], f"{what}: {name} statistics (events, errors, aggregates) {h[1]} != {c[1]}"
            # a real out-of-range index next to the holes: refused, nothing applied
            bad = holey.copy()
            bad[len(bad) // 2, 8:16] = np.array([n_agg], dtype=np.uint64).view(np.uint8)
            e.set_initial_states(None)
            e.fold_unsorted(base, n_agg)
            before = e.export_states()
            with pytest.raises(SgrError) as ei:
                e.fold_incremental(bad)
            assert ei.value.code == N.SGR_ERR_INVALID, f"{what}: {ei.value}"
            same(e.export_states()[:, :sb - 8], before[:, :sb - 8], f"{what}: refused batch left the program bytes")
            with pytest.raises(SgrError) as ei:
                e.load_unsorted(bad, n_agg)
            assert ei.value.code == N.SGR_ERR_INVALID, f"{what}: {ei.value}"


# ------------------------------------------------------------------ C. replay-list overflow of the record-parallel fold
def test_full_fold_with_more_throwing_aggregates_than_the_replay_list():
    """1.1 M aggregates, each with one throw at a random position: more throwing segments than the runs kernel's replay list
    holds, so the host re-runs the whole fold on the sequential kernel. Byte for byte against the C oracle."""
    n_agg = 1_100_000
    rng = np.random.default_rng(11)
    counts = rng.integers(1, 5, size=n_agg)
    n = int(counts.sum())
    starts = np.zeros(n_agg + 1, dtype=np.int64)
    np.cumsum(counts, out=starts[1:])
    agg = np.repeat(np.arange(n_agg, dtype=np.uint64), counts)
    types = rng.integers(0, 3, size=n).astype(np.uint32)
    types[starts[:-1] + rng.integers(0, counts)] = 3
    seqs = (np.arange(n) - np.repeat(starts[:-1], counts) + 1).astype(np.uint32)
    rec = _counter_records(agg, types, seqs, rng.integers(-2**31, 2**31, size=n).astype(np.int32))
    off = (starts * 64).astype(np.uint64)
    want, nev, nerr = O.fold_packed(O.MODEL_COUNTER, O.REC_FIXED64, rec, off, threads=8)
    assert nerr == n_agg > REDO_CAP
    with ReplayEngine(0) as e:
        e.register_program(P.counter_program())
        e.set_option("kernel", 0)
        e.load_events(rec, off)
        e.fold()
        st = e.stats()
        assert st.fold_launches == 2, "the overflow re-run did not happen"
        same(e.export_states(), want, "full fold after a replay-list overflow")
        assert (st.n_events, st.n_errors) == (nev, nerr)


@pytest.mark.parametrize("ingest", ["host", "device"])
def test_in_place_replay_overflow_invalidates_until_reset(ingest):
    """incremental=1: a poll of 2^20 + 1 new ids that all throw overflows the replay list of an in-place fold. The poll fails and
    the table is half-applied, so it must stay unreadable — get raises, the next poll fails with SGR_ERR_STATE, offsets stay —
    until the caller resets it; a rebuild from offset 0 then equals the oracle."""
    rng = np.random.default_rng(21)
    n1, n2 = 1000, REDO_CAP + 1
    ids1 = np.arange(n1, dtype=np.uint32)
    ids2 = np.arange(n1, n1 + n2, dtype=np.uint32)
    ids3 = rng.integers(0, n1, size=50).astype(np.uint32)
    parts = [(ids1, np.zeros(n1)), (ids2, np.full(n2, 3)), (ids3, rng.integers(0, 3, size=50))]
    wires, arrays, off = [], [], 0
    for a, t in parts:
        t = t.astype(np.uint32)
        s = np.arange(off + 1, off + len(a) + 1, dtype=np.uint32)
        b = rng.integers(-1000, 1000, size=len(a)).astype(np.int32)
        wires.append(O.kafka_encode_counter(a, t, s, b, recs_per_batch=512, lz4=True, base_offset=off).tobytes())
        arrays.append((a, t, s, b))
        off += len(a)
    with ReplayEngine(0) as e:
        e.register_program(P.counter_program())
        e.set_option("incremental", 1)
        if ingest == "device":
            dg = DeviceIngest(e, 1 << 21)

            def poll(w):
                dg.submit(0, w)
                dg.fold()

            def folded():
                return dg.offsets(0)[1]
        else:
            ing = Ingest()

            def poll(w):
                ing.record_batches(0, w)
                e.fold_ingested(ing)

            def folded():
                return ing.offsets(0)[1]
        poll(wires[0])
        assert folded() == n1
        with pytest.raises(SgrError) as ei:
            poll(wires[1])
        assert "replay list overflow" in str(ei.value), ei.value
        assert folded() == n1
        with pytest.raises(InvalidStateStoreException):
            e.get("agg-0")
        with pytest.raises(SgrError) as ei:
            poll(wires[2])
        assert ei.value.code == N.SGR_ERR_STATE, ei.value
        assert folded() == n1
        # reset and rebuild from offset 0 in one poll (the sort-free fold: no replay list)
        e.set_initial_states(None)
        e.set_option("incremental", 0)
        if ingest == "device":
            dg.reset()
            for w in wires:
                dg.submit(0, w)
            dg.fold()
            assert folded() == off
        else:
            ing = Ingest()
            for w in wires:
                ing.record_batches(0, w)
            e.fold_ingested(ing)
        n_keys = n1 + n2
        allrec = np.concatenate([_counter_records(*a) for a in arrays])
        want = O.fold_incremental(O.MODEL_COUNTER, allrec, np.zeros((n_keys, 16), dtype=np.uint8))
        got = e.export_states()
        assert not got[n_keys:].any()
        if ingest == "host":
            same(got[:n_keys], want, "rebuild after the overflow")
        else:
            # device indices follow no order: the table as a multiset of rows, and a sample of ids one by one
            same(np.unique(got[:n_keys], axis=0), np.unique(want, axis=0), "rebuild after the overflow (rows as a set)")
            for i in list(rng.integers(0, n_keys, size=3000)) + [0, n1 - 1, n_keys - 1]:
                j = e.index_of(f"agg-{i}")
                same(got[j:j + 1], want[i:i + 1], f"agg-{i} -> slot {j}")
            dg.close()


TOMBSTONE_THEN_THROW = {
    # class 1 (IF_EXISTS rules): the general record-parallel kernel
    "class1_16": (16, [(I.CREATE, [(I.OP_SET, 0, 16, 4), (I.OP_SET, 4, 20, 4)]), (I.IF_EXISTS, [(I.OP_ADD_I32, 0, 24, 4)]),
                       (I.TOMBSTONE, []), (I.THROW, [])]),
    # class 0 with 32- and 64-byte states: the wide kernels, which compose like class 1
    "class0_32": (32, [(I.CREATE, [(I.OP_SET, 0, 16, 8)]), (I.MATERIALISE, [(I.OP_ADD_I32, 8, 24, 4)]), (I.TOMBSTONE, []), (I.THROW, [])]),
    "class0_64": (64, [(I.CREATE, [(I.OP_SET, 0, 16, 16)]), (I.MATERIALISE, [(I.OP_ADD_I32, 40, 24, 4)]), (I.TOMBSTONE, []), (I.THROW, [])]),
}


@pytest.mark.parametrize("name", list(TOMBSTONE_THEN_THROW))
def test_throw_after_a_tombstone_in_another_lane(name):
    """A segment whose tombstone and throw land in different lanes of the record-parallel kernel: the throw's transformer has no
    exists-op, and composing it after the tombstoned prefix must keep its error bit (the state stays, ERROR, err_idx). Found by the
    device-ingest parity above, where it depended on the dense indices the decoder handed out."""
    sb, rules = TOMBSTONE_THEN_THROW[name]
    prog = P.make_program(sb, N.REC_FIXED64, rules)
    rng = np.random.default_rng(len(name) * 31 + sb)
    n_agg = 3000
    segs = []
    for a in range(n_agg):
        pre = list(rng.choice([0, 1], size=int(rng.integers(0, 9))))
        post = list(rng.integers(0, 4, size=int(rng.integers(0, 3))))
        segs.append(pre + [2, 3] + post if rng.random() < 0.8 else pre + post)
    counts = np.array([len(s) for s in segs])
    types = np.concatenate([np.asarray(s, dtype=np.uint32) for s in segs])
    n = len(types)
    rec = rng.integers(0, 256, size=(n, 64), dtype=np.uint8)
    rec[:, 0:4] = types.view(np.uint8).reshape(-1, 4)
    rec[:, 4:8] = np.arange(1, n + 1, dtype=np.uint32).view(np.uint8).reshape(-1, 4)
    rec[:, 8:16] = np.repeat(np.arange(n_agg, dtype=np.uint64), counts).view(np.uint8).reshape(-1, 8)
    off = np.zeros(n_agg + 1, dtype=np.uint64)
    np.cumsum(counts * 64, out=off[1:])
    want = I.fold(rules, sb, rec, off)
    with ReplayEngine(0) as e:
        e.register_program(prog)
        e.set_option("kernel", 2)                               # the record-parallel kernel, whatever the state width
        e.load_events(rec, off)
        e.fold()
        same(e.export_states(), want, f"{name}: full fold")
        e.set_option("kernel", 0)
        e.set_option("incremental", 1)                          # micro-batch onto a live table: the same kernel, in place
        e.set_initial_states(want)
        e.fold_incremental(rec)
        same(e.export_states(), I.fold_arrival_order(rules, sb, rec, want), f"{name}: in-place micro-batch")
