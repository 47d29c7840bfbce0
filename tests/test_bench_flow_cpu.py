"""bench.py's wire-format section, dry-run with stub engine / ingest / torch.distributed objects (no GPU): the section must leave a
result on every path — fine, set-up failure, failure inside the timed part — and under several ranks every rank must take part in
exactly one verdict exchange whatever happened to it (a barrier inside a try block would hang the ranks that did not fail).
The producer-side encoder runs for real on a small log."""
import re, sys, types, time, os
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
src = open(os.path.join(ROOT, 'bench.py')).read()
a = src.index("    wire_res = None\n    wire = {}")
b = src.index("    clocks = sampler.stop()")
block = "\n".join(l[4:] if l.startswith("    ") else l for l in src[a:b].splitlines())

class FakeTensor:
    def __init__(self, arr): self.arr = arr
    def view(self, *s): return FakeTensor(self.arr.reshape(*s))
    def __getitem__(self, k): return FakeTensor(self.arr[k])
    def cpu(self): return self
    def numpy(self): return self.arr
    def item(self): return int(self.arr.reshape(-1)[0])
class FakeTorch:
    uint8 = np.uint8; int32 = np.int32
    class cuda:
        @staticmethod
        def synchronize(): pass
    @staticmethod
    def empty(n, dtype=None, pin_memory=False): return FakeTensor(np.empty(n, dtype=np.uint8))
    @staticmethod
    def tensor(v, dtype=None, device=None): return FakeTensor(np.array(v))
class FakeDist:
    class ReduceOp: MIN = 0
    def __init__(self, other_ok): self.other_ok = other_ok; self.calls = 0
    def all_reduce(self, t, op=None):
        self.calls += 1
        t.arr[...] = min(int(t.arr.reshape(-1)[0]), 1 if self.other_ok else 0)

def run(case, world=1, other_ok=True, fail_setup=False, fail_timed=False):
    N_AGG, EPA = 4096, 4
    n_events = N_AGG * EPA
    rec_np = np.zeros((N_AGG * EPA, 16), dtype=np.uint32)
    rec_np[:, 2] = np.repeat(np.arange(N_AGG), EPA); rec_np[:, 1] = np.tile(np.arange(EPA), N_AGG); rec_np[:, 4] = 1
    state = {"steps": 0}
    class Eng:
        def __init__(self, *_): pass
        def register_program(self, p): pass
        def set_initial_states(self, s): pass
        def export_states(self, out): pass
        def get(self, k): return bytes(8)
        def states_tensor(self): return FakeTensor(np.zeros((N_AGG, 16), dtype=np.uint8))
        def close(self): state["closed_e"] = True
    class DG:
        def __init__(self, e, n):
            if fail_setup: raise RuntimeError("boom in set-up")
        def reset(self): pass
        def submit(self, p, t): pass
        def fold(self):
            state["steps"] += 1
            if fail_timed and state["steps"] > 2: raise RuntimeError("boom in timed part")
            return {"n_records": n_events, "n_new_keys": N_AGG, "n_decompressed_bytes": 1, "n_batches": 2}
        def last_timing(self): return {}
        def close(self): state["closed_dg"] = True
    fake_dingest = types.ModuleType("surge_b200.dingest"); fake_dingest.DeviceIngest = DG
    sys.modules["surge_b200.dingest"] = fake_dingest
    ns = dict(os=os, time=time, np=np, torch=FakeTorch, dist=FakeDist(other_ok), world=world, dev="cpu", local_rank=0,
              rec=FakeTensor(rec_np), N_AGG=N_AGG, EVENTS_PER_AGG=EPA, n_events=n_events, ke=3, host_states_np=None,
              ReplayEngine=Eng, P=types.SimpleNamespace(counter_program=lambda: None), eng=Eng(), note=lambda m: None)
    os.environ.pop("SGR_BENCH_SKIP_WIRE", None)
    exec(compile(block, "wire_section", "exec"), ns)
    res = ns["wire_res"]
    assert ns["dist"].calls == (1 if world > 1 else 0), case          # every rank, exactly once
    assert ("closed_dg" in state) == (not fail_setup), case               # what was opened is closed
    return res



def test_wire_section_leaves_a_result_on_every_path():
    saved = sys.modules.get("surge_b200.dingest")
    try:
        assert "seconds" in run("single rank, all fine")
        assert "error" in run("single rank, set-up fails", fail_setup=True)
        assert "error" in run("single rank, timed part fails", fail_timed=True)
        assert "seconds" in run("8 ranks, all fine", world=8)
        assert "another rank" in run("8 ranks, another rank failed", world=8, other_ok=False)["error"]
        assert "boom" in run("8 ranks, this rank failed", world=8, fail_setup=True)["error"]
    finally:
        if saved is not None:
            sys.modules["surge_b200.dingest"] = saved
        else:
            sys.modules.pop("surge_b200.dingest", None)


def test_dumped_state_columns_keep_every_32_bit_word(tmp_path):
    """--dump-outputs: count and version are signed, flags and err_idx unsigned, all exact in float64, and the file reads back."""
    import pytest
    import bench

    tab = np.zeros((3, 16), dtype=np.uint8)
    tab.view(np.int32)[0] = [-(1 << 31), 7, 3, 0]
    tab.view(np.uint32)[1] = [0xFFFFFFFF, 1 << 31, 0xFFFFFFFF, 5]
    cols = bench.state_columns(tab)
    assert cols.dtype == np.float64
    assert cols.tolist() == [[-(1 << 31), 7, 3, 0], [-1, -(1 << 31), 0xFFFFFFFF, 5], [0, 0, 0, 0]]
    bench.dump_outputs(str(tmp_path), {"states": cols})
    assert np.array_equal(np.load(tmp_path / "states.npy"), cols)
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path), {"states": np.zeros(bench.DUMP_MAX_BYTES // 8 + 1)})
