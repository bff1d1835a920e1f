"""The reference's own native kernels (oracle/_ref/libjvector.so) for the tests that pin the oracle and the legacy C ABI
against them, recorded call by call under tests/golden/reference/<test module>.npz so that those tests need nothing
outside this repository.

By default the `ref` fixture is a `Replay`: each call must come in the recorded order with the recorded scalar arguments;
it writes what the reference wrote through its output pointers and returns what the reference returned. A test's
assertions are therefore the same whether the reference runs or its answers are read back. With JV_RECORD_REFERENCE=1
(where oracle_lib.build() can build the library from the reference's sources) the fixture is a `Recorder` that runs the
real library, and the session rewrites the recordings of the tests it ran."""
import ctypes as C
import os

import numpy as np

import oracle_lib as o

GOLDEN = os.path.join(o.GOLDEN, "reference")
RECORD = os.environ.get("JV_RECORD_REFERENCE") == "1"

# kernels that write through a pointer: name -> (argument index, first element written, element count), from the call's arguments
WRITES = {
    "add_in_place_f32": (0, lambda a: 0, lambda a: a[2]),
    "sub_in_place_f32": (0, lambda a: 0, lambda a: a[2]),
    "min_in_place_f32": (0, lambda a: 0, lambda a: a[2]),
    "add_scalar_in_place_f32": (0, lambda a: 0, lambda a: a[2]),
    "sub_scalar_in_place_f32": (0, lambda a: 0, lambda a: a[2]),
    "nvq_shuffle_query_in_place_8bit": (0, lambda a: 0, lambda a: a[1]),
    "nvq_quantize_8bit": (6, lambda a: 0, lambda a: a[1]),
    "calculate_partial_sums_dot_f32": (6, lambda a: a[1] * a[3], lambda a: a[3]),
    "calculate_partial_sums_euclidean_f32": (6, lambda a: a[1] * a[3], lambda a: a[3]),
    "calculate_partial_sums_self_magnitude_f32": (4, lambda a: a[1] * a[3], lambda a: a[3]),
}
# The LUT rows of the partial-sum kernels are recorded for the first SAMPLED_CODEBOOKS subspaces only (every subspace width the
# tests use occurs among them) and replayed as NaN elsewhere: a whole M = 96 x 256 LUT per kernel would be most of the recording.
# Tests compare those outputs where they are not NaN; the sums the reference formed from the whole LUT are recorded in full.
SAMPLED_CODEBOOKS = 3
_SAMPLED = {"calculate_partial_sums_dot_f32", "calculate_partial_sums_euclidean_f32", "calculate_partial_sums_self_magnitude_f32"}


def _recorded(name, args):
    return name not in _SAMPLED or int(args[1]) < SAMPLED_CODEBOOKS


def where_recorded(lut):
    """entries of a partial-sum LUT the reference filled (all of them when it runs, the sampled subspaces on replay)"""
    m = ~np.isnan(lut)
    assert m.any()
    return m


_DTYPES = {o.f32p: np.float32, o.u8p: np.uint8}


def _scalars(name, args):
    _, types = o.REF_SIGNATURES[name]
    return [float(a) for a, t in zip(args, types) if t not in _DTYPES]


def _written(name, args):
    """numpy view of the elements `name` writes through its output pointer (None when it writes none)"""
    if name not in WRITES:
        return None
    i, first, count = WRITES[name]
    f, n = int(first(args)), int(count(args))
    return np.ctypeslib.as_array(args[i], shape=(f + n,))[f:]


def _ret_bits(restype, value):
    if restype is None:
        return 0
    if restype is C.c_float:
        return int(np.float64(value).view(np.int64))
    return int(value)


def _ret_value(restype, bits):
    if restype is None:
        return None
    if restype is C.c_float:
        return float(np.int64(bits).view(np.float64))
    return int(bits)


class Recorder:
    """Runs the reference library and records each call of one test."""

    def __init__(self, lib):
        self._lib = lib
        self.names, self.args, self.rets, self.f32, self.u8, self.captures = [], [], [], [], [], []

    def __getattr__(self, name):
        if name not in o.REF_SIGNATURES:
            raise AttributeError(name)

        def call(*args):
            value = getattr(self._lib, name)(*args)
            self.names.append(name)
            self.args += _scalars(name, args)
            self.rets.append(_ret_bits(o.REF_SIGNATURES[name][0], value))
            out = _written(name, args)
            if out is not None and _recorded(name, args):
                (self.f32 if out.dtype == np.float32 else self.u8).append(out.copy())
            return value
        return call

    def capture(self, compute):
        """a value the test derives from the reference library by other means (its symbol table, the oracle routed through it)"""
        value = np.asarray(compute())
        self.captures.append(value)
        return value

    def arrays(self):
        d = {"names": np.array(self.names, dtype=str), "args": np.array(self.args, np.float64), "rets": np.array(self.rets, np.int64),
             "f32": np.concatenate(self.f32) if self.f32 else np.empty(0, np.float32),
             "u8": np.concatenate(self.u8) if self.u8 else np.empty(0, np.uint8)}
        d.update({"capture%d" % i: v for i, v in enumerate(self.captures)})
        return d


# One .npz per test module: each field of every test's recording concatenated over the tests (with per-test lengths), and the
# captures of a test as "<test>|capture<i>".
FIELDS = ("names", "args", "rets", "f32", "u8")


def _pack(tests):
    names = sorted(tests)
    out = {"tests": np.array(names, dtype=str)}
    for f in FIELDS:
        out[f] = np.concatenate([tests[t][f] for t in names])
        out["len_" + f] = np.array([len(tests[t][f]) for t in names], np.int64)
    for t in names:
        out.update({"%s|%s" % (t, k): v for k, v in tests[t].items() if k not in FIELDS})
    return out


def _unpack(arrays):
    tests = {str(t): {} for t in arrays["tests"]}
    for f in FIELDS:
        lens = arrays["len_" + f]
        for t, end, n in zip(arrays["tests"], np.cumsum(lens), lens):
            tests[str(t)][f] = arrays[f][end - n:end]
    for k, v in arrays.items():
        if "|" in k:
            t, f = k.split("|", 1)
            tests[t][f] = v
    return tests


_loaded = {}


def _load(module):
    """{test: {field: array}} of one test module's recording"""
    if module not in _loaded:
        path = os.path.join(GOLDEN, module + ".npz")
        _loaded[module] = _unpack(dict(np.load(path, allow_pickle=False))) if os.path.exists(path) else {}
    return _loaded[module]


class Replay:
    """Reads back what the reference returned and wrote, call for call, for one test."""

    def __init__(self, module, test):
        rec = _load(module)
        if test not in rec:
            raise AssertionError("no recorded reference answers for %s::%s under %s: record them with JV_RECORD_REFERENCE=1 "
                                 "where oracle/_ref/libjvector.so can be built" % (module, test, GOLDEN))
        self._test = test
        self._rec = rec[test]
        self._call = self._arg = self._f32 = self._u8 = self._capture = 0

    def __getattr__(self, name):
        if name not in o.REF_SIGNATURES:
            raise AttributeError(name)

        def call(*args):
            names, i = self._rec["names"], self._call
            assert i < len(names), "%s: call %d (%s) was not recorded" % (self._test, i, name)
            assert names[i] == name, "%s: call %d is %s, the recording has %s" % (self._test, i, name, names[i])
            sc = _scalars(name, args)
            want = self._rec["args"][self._arg:self._arg + len(sc)].tolist()
            assert sc == want, "%s: call %d %s has scalar arguments %s, the recording %s" % (self._test, i, name, sc, want)
            out = _written(name, args)
            if out is not None and not _recorded(name, args):
                out[:] = np.nan
            elif out is not None:
                src, pos = ("f32", self._f32) if out.dtype == np.float32 else ("u8", self._u8)
                out[:] = self._rec[src][pos:pos + len(out)]
                if src == "f32":
                    self._f32 += len(out)
                else:
                    self._u8 += len(out)
            self._call, self._arg = i + 1, self._arg + len(sc)
            return _ret_value(o.REF_SIGNATURES[name][0], self._rec["rets"][i])
        return call

    def capture(self, compute):
        value = self._rec["capture%d" % self._capture]
        self._capture += 1
        return value


def save(recorded):
    """merge {module: {test: {field: array}}} into the golden recordings"""
    os.makedirs(GOLDEN, exist_ok=True)
    for module, tests in recorded.items():
        merged = dict(_load(module), **tests)
        np.savez_compressed(os.path.join(GOLDEN, module + ".npz"), **_pack(merged))
