"""The argument contract of the fifteen orbx_match_hamming* entry points, pinned as a table.

Every entry point starts from a valid call on small buffers, and the grid applies one perturbation at a time: each pointer
NULL; each size -1, 0 and the first value past its limit (2^20 rows, 65536 sets, k = 0 and 33, cap -1); max_distance 0,
FLT_EPSILON, NaN and +inf.  It also runs every (size 0, pointer NULL) and every (limit exceeded, pointer NULL) pair, since
those are where the forms check in different orders.  Each call records its return code, the launches it queued, and
where the entry point has them the host *n_out, the host offsets and the device d_n_out / d_offsets, each pre-filled with
a sentinel (a list trimmed of trailing sentinels: [] = untouched).

The expected table is `match_entry_contract.json`.  A deliberate change of a check order or a return code shows up as a
diff of that table: regenerate it on a GPU with `python tests/test_match_entry_contract.py`.

Every buffer is as large as the largest size any call of the grid passes (the host train buffer holds the 2 x 2^20 rows
that orbx_match_hamming_sets uploads before it rejects the stride), so no call the library accepts reads or writes past
a buffer.
"""
import ctypes as C
import functools
import json
import os
import sys

import numpy as np
import pytest

TABLE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "match_entry_contract.json")
OK, E_ARG, E_UNSUPPORTED = 0, -1, -5
ROWS_PAST, SETS_PAST = 1 << 20, 65536
FLT_EPS = float(np.finfo(np.float32).eps)
SENT = -0x5A5A5A5                     # sentinel of every recorded output
WINDOW = 16                           # recorded entries of an offsets / n_out array
BASE = {"rows": 3, "train": 5, "sets": 2, "k": 3, "cap": 64, "md": 120.0}

# Buffer sizes (bytes or entries) that hold every accepted call of the grid: one size at its largest, the others at BASE.
HQ_BYTES = ROWS_PAST * 32                                  # host query: 2^20 rows
HT_BYTES = 2 * ROWS_PAST * 32                              # host train: 2 sets x 2^20 rows (_sets uploads it, then rejects)
HBEST_BYTES = ROWS_PAST * 4 * 16                           # knn k = 3 / knn2 [nq][2] / sets [2][nq] at nq = 2^20
DQ_BYTES = 2 * ROWS_PAST * 32
DT_BYTES = 2 * ROWS_PAST * 32
DBEST_BYTES = ROWS_PAST * 2 * 4 * 16                       # device knn k = 3, 2 sets, nq = 2^20
OFF_ENTRIES = 2 * ROWS_PAST + 2                            # 2 sets x 2^20 lists + 1

# Entry points: (name, [(argument, kind)]).  Pointer kinds name the buffer (h*: host, d*: device); the other kinds are
# rows / train (a row count or stride), sets, k, cap and md (max_distance).
Q, T = ("q", "hq"), ("t", "ht")
DQ, DT, DTC, DQC = ("d_query", "dq"), ("d_train", "dt"), ("d_train_counts", "dtcounts"), ("d_query_counts", "dqcounts")
PW = [DQ, ("query_stride", "rows"), DQC, DT, ("train_stride", "train"), DTC, ("npairs", "sets")]
RG = [DQ, ("nq", "rows"), DT, ("train_stride", "train"), DTC, ("nsets", "sets")]
ENTRIES = [
    ("orbx_match_hamming", [Q, ("nq", "rows"), T, ("nt", "train"), ("out", "hbest"), ("n_out", "hnout")]),
    ("orbx_match_hamming_knn2", [Q, ("nq", "rows"), T, ("nt", "train"), ("out", "hbest"), ("n_out", "hnout")]),
    ("orbx_match_hamming_knn", [Q, ("nq", "rows"), T, ("nt", "train"), ("k", "k"), ("out", "hbest"), ("n_out", "hnout")]),
    ("orbx_match_hamming_crosscheck", [Q, ("nq", "rows"), T, ("nt", "train"), ("out", "hbest"), ("n_out", "hnout")]),
    ("orbx_match_hamming_sets", [Q, ("nq", "rows"), T, ("train_stride", "train"), ("train_counts", "hcounts"), ("nsets", "sets"),
                                 ("best", "hbest"), ("second", "hsecond")]),
    ("orbx_match_hamming_radius", [Q, ("nq", "rows"), T, ("nt", "train"), ("max_distance", "md"), ("out", "hbest"), ("cap", "cap"),
                                   ("offsets", "hoff"), ("n_out", "hnout")]),
    ("orbx_match_hamming_device", [DQ, ("nq", "rows"), DT, ("nt", "train"), ("nsets", "sets"), ("d_best", "dbest"),
                                   ("d_second", "dsecond")]),
    ("orbx_match_hamming_device_ragged", RG + [("d_best", "dbest"), ("d_second", "dsecond")]),
    ("orbx_match_hamming_device_crosscheck", RG + [("d_out", "dbest"), ("d_n_out", "dnout")]),
    ("orbx_match_hamming_device_knn", RG + [("k", "k"), ("d_out", "dbest")]),
    ("orbx_match_hamming_device_radius", RG + [("max_distance", "md"), ("d_out", "dbest"), ("cap", "cap"), ("d_offsets", "doff")]),
    ("orbx_match_hamming_device_pairwise", PW + [("d_best", "dbest"), ("d_second", "dsecond")]),
    ("orbx_match_hamming_device_pairwise_crosscheck", PW + [("d_out", "dbest"), ("d_n_out", "dnout")]),
    ("orbx_match_hamming_device_pairwise_knn", PW + [("k", "k"), ("d_out", "dbest")]),
    ("orbx_match_hamming_device_pairwise_radius", PW + [("max_distance", "md"), ("d_out", "dbest"), ("cap", "cap"),
                                                        ("d_offsets", "doff")]),
]
SIZE_VALUES = {"rows": (-1, 0, ROWS_PAST), "train": (-1, 0, ROWS_PAST), "sets": (-1, 0, SETS_PAST), "k": (-1, 0, 33), "cap": (-1, 0)}
PAST_LIMIT = {"rows": (ROWS_PAST,), "train": (ROWS_PAST,), "sets": (SETS_PAST,), "k": (0, 33), "cap": (-1,)}
MD_VALUES = (0.0, FLT_EPS, float("nan"), float("inf"))
RECORDED = ("hnout", "hoff", "dnout", "doff")              # the outputs a call's record holds, in this order


def is_pointer(kind):
    return kind[0] in "hd" and kind not in SIZE_VALUES


def grid(args):
    """The perturbations of one entry point: a list of {argument: value} (value None: a NULL pointer)."""
    ptrs = [a for a, k in args if is_pointer(k)]
    cases = [{}]
    for a, k in args:
        if is_pointer(k):
            cases.append({a: None})
        elif k in SIZE_VALUES:
            cases += [{a: v} for v in SIZE_VALUES[k]]
        elif k == "md":
            cases += [{a: v} for v in MD_VALUES]
    for a, k in args:
        if k in SIZE_VALUES:
            for v in sorted(set((0,) + PAST_LIMIT[k])):
                cases += [{a: v, p: None} for p in ptrs]
    return cases


def case_id(case):
    return ",".join(f"{a}={'NULL' if v is None else v}" for a, v in case.items()) or "base"


def is_empty(args, case):
    """A row count, stride or set count of 0: no work to do."""
    sizes = {a: case.get(a, BASE[k]) for a, k in args if k in ("rows", "train", "sets")}
    return 0 in sizes.values()


@functools.lru_cache(maxsize=None)
def load_table():
    with open(TABLE) as f:
        return json.load(f)


def test_table_covers_the_grid():
    """The table holds one record for every case of every entry point's grid, and nothing else."""
    table = load_table()
    assert sorted(table) == sorted(n for n, _ in ENTRIES)
    for name, args in ENTRIES:
        assert sorted(table[name]) == sorted(case_id(c) for c in grid(args)), name
        nrec = 2 + sum(k in RECORDED for _, k in args)
        assert all(len(r) == nrec for r in table[name].values()), name


def test_rejected_and_empty_calls_launch_nothing():
    """An argument error or an empty input is reported before anything is queued on the GPU."""
    for name, args in ENTRIES:
        for c in grid(args):
            rc, launches = load_table()[name][case_id(c)][:2]
            if rc in (E_ARG, E_UNSUPPORTED) or is_empty(args, c):
                assert launches == 0, (name, case_id(c), rc)


class Buffers:
    """One context and every buffer of the grid, host and device, filled with seeded random descriptors."""

    def __init__(self):
        import torch
        from rgbd_visualodometry_b200 import orb
        self.torch = torch
        self.ctx = orb.Context(1, 1.2, 1, 64, 64, 1)
        rng = np.random.default_rng(20261022)
        self.host = {
            "hq": rng.integers(0, 256, HQ_BYTES, dtype=np.uint8),
            "ht": rng.integers(0, 256, HT_BYTES, dtype=np.uint8),
            "hbest": np.zeros(HBEST_BYTES, np.uint8),
            "hsecond": np.zeros(HBEST_BYTES // 2, np.uint8),
            "hcounts": np.resize(np.array([BASE["train"], BASE["train"] - 1], np.int32), SETS_PAST),
            "hoff": np.zeros(ROWS_PAST + 2, np.int64),
        }
        g = torch.Generator(device="cuda").manual_seed(20261022)
        rand = lambda n: torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=g)  # noqa: E731
        self.dev = {
            "dq": rand(DQ_BYTES), "dt": rand(DT_BYTES),
            "dbest": torch.zeros(DBEST_BYTES, dtype=torch.uint8, device="cuda"),
            "dsecond": torch.zeros(DBEST_BYTES // 2, dtype=torch.uint8, device="cuda"),
            "dtcounts": torch.tensor([BASE["train"], BASE["train"] - 1], dtype=torch.int32, device="cuda").repeat(SETS_PAST // 2),
            "dqcounts": torch.tensor([BASE["rows"], BASE["rows"] - 1], dtype=torch.int32, device="cuda").repeat(SETS_PAST // 2),
            "dnout": torch.zeros(SETS_PAST, dtype=torch.int32, device="cuda"),
            "doff": torch.zeros(OFF_ENTRIES, dtype=torch.int64, device="cuda"),
        }
        self.nout = C.c_int(0)
        torch.cuda.synchronize()

    def close(self):
        self.ctx.close()

    def value(self, kind, v):
        if v is None:
            return None
        if kind == "hnout":
            return C.byref(self.nout)
        if kind in self.host:
            return self.host[kind].ctypes.data
        if kind in self.dev:
            return self.dev[kind].data_ptr()
        return v

    def run(self, name, args, case):
        """One call of the grid -> [rc, launches, the recorded outputs the entry point has]."""
        torch = self.torch
        self.nout.value = SENT
        self.host["hoff"][:WINDOW] = SENT
        self.dev["dnout"][:WINDOW].fill_(SENT)
        self.dev["doff"][:WINDOW].fill_(SENT)
        torch.cuda.synchronize()
        vals = [self.value(k, case.get(a, BASE.get(k, "buffer"))) for a, k in args]
        lib = self.ctx.lib
        before = self.ctx.launch_count
        rc = getattr(lib, name)(self.ctx.h, *vals)
        self.ctx.synchronize()
        rec = [rc, self.ctx.launch_count - before]
        for k in RECORDED:
            if any(kind == k for _, kind in args):
                if k == "hnout":
                    rec.append(self.nout.value)
                else:
                    w = self.host[k][:WINDOW] if k in self.host else self.dev[k][:WINDOW].cpu().numpy()
                    rec.append(trimmed(w))
        return rec


def trimmed(w):
    w = [int(x) for x in w]
    while w and w[-1] == SENT:
        w.pop()
    return w


def run_grid(bufs, name, args):
    return {case_id(c): bufs.run(name, args, c) for c in grid(args)}


@pytest.fixture(scope="module")
def bufs():
    b = Buffers()
    yield b
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n, _ in ENTRIES])
def test_entry_contract(bufs, name):
    args = dict(ENTRIES)[name]
    want = load_table()[name]
    got = run_grid(bufs, name, args)
    diff = {c: (got[c], want.get(c)) for c in got if got[c] != want.get(c)}
    assert not diff, f"{name}: {len(diff)} cases differ from the table (got, want): {diff}"


def write_table(path=TABLE):
    bufs = Buffers()
    try:
        table = {name: run_grid(bufs, name, args) for name, args in ENTRIES}
    finally:
        bufs.close()
    with open(path, "w") as f:                               # one case per line, so that a change is a small diff
        f.write("{\n")
        for i, (name, cases) in enumerate(table.items()):
            f.write(f"  {json.dumps(name)}: {{\n")
            lines = [f"    {json.dumps(c)}: {json.dumps(r)}" for c, r in cases.items()]
            f.write(",\n".join(lines) + ("\n  }" + (",\n" if i + 1 < len(table) else "\n")))
        f.write("}\n")


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    write_table(sys.argv[1] if len(sys.argv) > 1 else TABLE)
