"""The reference's own SIMD loops (oracle/_ref/libarrowgo_ref.so), recorded once and replayed.

oracle/Makefile assembles oracle/_ref from the original project's sources, which only a development machine has.
Elsewhere the `ref` fixture hands the tests a Replay instead.  The calls each test makes to the reference were
recorded in order into a running digest of every call's function name, scalar arguments, input bytes and the output
bytes the reference produced; the digest is stored every CHECK_EVERY calls and after the test's last call.  The
recording also keeps the output itself wherever the C restatement (oracle/cpu_ref.c) or a bit model below does not
reproduce it, and for scalar results.  On replay the output is that stored value or the restatement's answer, and a
call that completes a checkpoint raises unless the running digest equals the recorded one.  So a test that compares
against `ref` still compares against the reference's bits.

To record, on a machine where oracle/_ref builds and with a GPU for the GPU tests:

    AG_REF_RECORD=tests/golden/ref_replay.npz python -m pytest tests
"""
import atexit
import ctypes as C
import hashlib
import os

import numpy as np

from arrow_go_b200 import _native as N
from helpers import NP_OF, TYPE_NAME

RECORD_ENV = "AG_REF_RECORD"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_replay.npz")

SZ = {t: np.dtype(d).itemsize for t, d in NP_OF.items()}
TYPE_OF = {nm: t for t, nm in TYPE_NAME.items()}
CMP = {"equal": N.CMP_EQ, "not_equal": N.CMP_NE, "greater": N.CMP_GT, "greater_equal": N.CMP_GE}
SHAPE = {"arr_arr": N.SHAPE_AA, "arr_scalar": N.SHAPE_AS, "scalar_arr": N.SHAPE_SA}
BITOP = {"and": N.BITOP_AND, "or": N.BITOP_OR, "xor": N.BITOP_XOR, "and_not": N.BITOP_ANDNOT}
ARITH_SHAPE = {"arithmetic_binary": N.SHAPE_AA, "arithmetic_arr_scalar": N.SHAPE_AS, "arithmetic_scalar_arr": N.SHAPE_SA}

# entry points whose prototypes oracle.ref() leaves to the tests
PROTOTYPES = {
    "unpack32_avx2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "bytes_to_bools_avx2": (None, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "bytes_to_bools_sse4": (None, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "levels_to_bitmap_bmi2": (C.c_uint64, [C.c_void_p, C.c_int, C.c_int16]),
}


class Call:
    """One call: its scalar arguments, the (address, size) regions it reads and writes, and a function that computes
    the same outputs (and return value) without the reference, or None."""

    def __init__(self, scalars, inputs, outputs, produce=None, returns=False):
        self.scalars, self.inputs, self.outputs, self.produce, self.returns = scalars, inputs, outputs, produce, returns


def _read(region):
    addr, nbytes = region
    return C.string_at(addr, nbytes) if nbytes > 0 else b""


def _write(region, data):
    if region[1] > 0:
        C.memmove(region[0], data, region[1])


def _unpack32_model(src, dst, n, bits):
    """value i = bits [i*b, (i+1)*b) of the little-endian stream, whole groups of 32 values only"""
    n = n // 32 * 32
    if n:
        words = np.frombuffer(C.string_at(src, n * bits // 8), dtype=np.uint8) if bits else np.zeros(0, np.uint8)
        stream = np.unpackbits(words, bitorder="little")
        out = np.zeros(n, dtype=np.uint64)
        for j in range(bits):
            out |= stream[np.arange(n) * bits + j].astype(np.uint64) << np.uint64(j)
        C.memmove(dst, out.astype(np.uint32).tobytes(), n * 4)
    return n


def _bytes_to_bools_model(src, length, dst, outlen):
    k = min(outlen, length * 8)
    if k:
        C.memmove(dst, np.unpackbits(np.frombuffer(C.string_at(src, length), np.uint8), bitorder="little")[:k].tobytes(), k)


def describe(name, args, cpu):
    """The Call of reference entry point `name` with `args` (SysV prototypes as oracle.ref() declares them)."""
    base = name.rsplit("_", 1)[0]
    if base in ("sum_float64", "sum_int64", "sum_uint64"):
        x, n, out = args
        return Call((n,), [(x, 8 * n)], [(out, 8)])
    if base in ARITH_SHAPE:
        t, op, l, r, out, n = args
        shape = ARITH_SHAPE[base]
        ln, rn = (1 if shape == N.SHAPE_SA else n), (1 if shape == N.SHAPE_AS else n)
        return Call((t, op, n), [(l, ln * SZ[t]), (r, rn * SZ[t])], [(out, n * SZ[t])],
                    lambda: cpu.ref_arith_binary(t, op, shape, l, r, out, n))
    if base == "arithmetic_unary_same_types":
        t, op, x, out, n = args
        return Call((t, op, n), [(x, n * SZ[t])], [(out, n * SZ[t])], lambda: cpu.ref_arith_unary_same(t, op, x, out, n))
    if base == "arithmetic_unary_diff_type":
        it, ot, op, x, out, n = args
        return Call((it, ot, op, n), [(x, n * SZ[it])], [(out, n * SZ[ot])],
                    lambda: cpu.ref_arith_unary_diff(it, ot, op, x, out, n))
    if base.endswith("_max_min"):
        t = TYPE_OF[base[:-len("_max_min")]]
        x, n, lo, hi = args
        return Call((n,), [(x, n * SZ[t])], [(lo, SZ[t]), (hi, SZ[t])])
    if base == "cast_type_numeric":
        it, ot, x, out, n = args
        return Call((it, ot, n), [(x, n * SZ[it])], [(out, n * SZ[ot])],
                    lambda: cpu.ref_cast_numeric(it, ot, x, None, 0, out, n, 1, 1, C.byref(C.c_int64())))
    if base.startswith("comparison_"):
        op, shape = next((o, s) for o in CMP for s in SHAPE if base == f"comparison_{o}_{s}")
        t, l, r, out, n, off = args
        ln, rn = (1 if SHAPE[shape] == N.SHAPE_SA else n), (1 if SHAPE[shape] == N.SHAPE_AS else n)
        nb = (off + n + 7) // 8
        return Call((t, n, off), [(l, ln * SZ[t]), (r, rn * SZ[t]), (out, nb)], [(out, nb)],
                    lambda: cpu.ref_compare(t, CMP[op], SHAPE[shape], l, r, out, n, off))
    if base.startswith("bitmap_aligned_"):
        op = BITOP[base[len("bitmap_aligned_"):]]
        l, r, out, nb = args
        return Call((nb,), [(l, nb), (r, nb)], [(out, nb)], lambda: cpu.ref_bitmap_op(op, l, 0, r, 0, out, 0, nb * 8))
    if base == "unpack32":
        src, dst, n, bits = args
        m = n // 32 * 32
        return Call((n, bits), [(src, m * bits // 8)], [(dst, m * 4)], lambda: _unpack32_model(src, dst, n, bits), True)
    if base == "bytes_to_bools":
        src, length, dst, outlen = args
        return Call((length, outlen), [(src, length), (dst, outlen)], [(dst, outlen)],
                    lambda: _bytes_to_bools_model(src, length, dst, outlen))
    if base == "levels_to_bitmap":
        lv, num, rhs = args
        return Call((num, rhs), [(lv, 2 * num)], [], returns=True)
    raise NotImplementedError(f"no replay description of reference entry point {name}")


CHECK_EVERY = 64  # calls per checkpoint of a test's running digest; its last call is one too


def _chain(state, name, call, ins, outs, ret):
    """The running digest of a test's calls, `state`, after one more call."""
    h = hashlib.blake2b(state, digest_size=8)
    h.update(f"{name}{call.scalars}{ret}".encode())
    for b in ins + outs:
        h.update(len(b).to_bytes(8, "little"))
        h.update(b)
    return h.digest()


def _is_check(j, count):
    return (j + 1) % CHECK_EVERY == 0 or j == count - 1


def _encode_ret(ret):
    return b"" if ret is None else (int(ret) % (1 << 64)).to_bytes(8, "little")


def key_of(node):
    """Stable across rootdirs and invocations: file name and test name with its parameters."""
    return f"{node.path.name}::{node.name}"


class _Fn:
    """A callable that, like a ctypes function, accepts restype / argtypes assignments."""

    def __init__(self, fn):
        self._fn = fn

    def __call__(self, *args):
        return self._fn(*args)


# ------------------------------------------------------------------------------------------------ recording ----
_recorded = {}
_recorded_isa = []
_functions = set()


def _save(path):
    keys = sorted(_recorded)
    calls = [c for k in keys for c in _recorded[k]]
    checks = [c[0] for k in keys for j, c in enumerate(_recorded[k]) if _is_check(j, len(_recorded[k]))]
    raw = [c[1] for c in calls]
    np.savez_compressed(
        path, isa=np.array(_recorded_isa[0]), functions=np.array(sorted(_functions)),
        tests=np.array(keys), counts=np.array([len(_recorded[k]) for k in keys], dtype=np.int32),
        checks=np.frombuffer(b"".join(checks), dtype=np.uint64),
        raw_len=np.array([-1 if r is None else len(r) for r in raw], dtype=np.int32),
        raw=np.frombuffer(b"".join(r for r in raw if r is not None), dtype=np.uint8))


class Recorder:
    """The live library, recording every call of one test."""

    def __init__(self, lib, key, cpu, isa):
        if not _recorded_isa:
            _recorded_isa.append(isa)
            atexit.register(_save, os.environ[RECORD_ENV])
        for fname, (restype, argtypes) in PROTOTYPES.items():
            if hasattr(lib, fname):
                getattr(lib, fname).restype, getattr(lib, fname).argtypes = restype, argtypes
        self._lib, self._cpu, self._calls = lib, cpu, _recorded.setdefault(key, [])
        self._state = bytes(8)

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def record(*args):
            _functions.add(name)
            call = describe(name, args, self._cpu)
            ins = [_read(r) for r in call.inputs]
            before = [_read(r) for r in call.outputs]
            ret = fn(*args)
            outs = [_read(r) for r in call.outputs]
            same = False
            if call.produce is not None:
                for r, b in zip(call.outputs, before):
                    _write(r, b)
                pret = call.produce()
                same = [_read(r) for r in call.outputs] == outs and (not call.returns or pret == ret)
                for r, b in zip(call.outputs, outs):
                    _write(r, b)
            ret = ret if call.returns else None
            self._state = _chain(self._state, name, call, ins, outs, ret)
            self._calls.append((self._state, None if same else b"".join(outs) + _encode_ret(ret)))
            return ret
        return _Fn(record)


# ------------------------------------------------------------------------------------------------ replay -------
_table = None


def table():
    global _table
    if _table is None:
        g = np.load(GOLDEN)
        counts = g["counts"].astype(np.int64)
        starts = np.concatenate([[0], np.cumsum(counts)])
        check_starts = np.concatenate([[0], np.cumsum((counts + CHECK_EVERY - 1) // CHECK_EVERY)])
        raw_len = g["raw_len"]
        _table = {"isa": str(g["isa"]), "functions": set(g["functions"].tolist()), "raw": g["raw"].tobytes(),
                  "checks": g["checks"].tobytes(), "raw_len": raw_len,
                  "raw_off": np.concatenate([[0], np.cumsum(np.maximum(raw_len, 0))]),
                  "tests": {k: (int(starts[i]), int(counts[i]), int(check_starts[i])) for i, k in enumerate(g["tests"].tolist())}}
    return _table


class Replay:
    """Stands in for the live library in one test, replaying that test's recorded calls in order."""

    def __init__(self, key, cpu):
        t = table()
        if key not in t["tests"]:
            raise LookupError(f"{key}: no recorded reference calls in {GOLDEN}; record them (see {__file__})")
        self._t, self._key, self._cpu = t, key, cpu
        self._first, self._count, self._check = t["tests"][key]
        self._j, self._state = 0, bytes(8)

    def __getattr__(self, name):
        if name not in self._t["functions"]:
            raise AttributeError(name)
        return _Fn(lambda *args: self._replay(name, args))

    def _replay(self, name, args):
        t, j = self._t, self._j
        if j >= self._count:
            raise AssertionError(f"{self._key}: call #{j} ({name}): the recording has only {self._count} calls")
        self._j += 1
        i = self._first + j
        call = describe(name, args, self._cpu)
        ins = [_read(r) for r in call.inputs]
        ret = None
        if t["raw_len"][i] >= 0:
            raw = t["raw"][t["raw_off"][i]:t["raw_off"][i] + t["raw_len"][i]]
            pos = 0
            for r in call.outputs:
                _write(r, raw[pos:pos + r[1]])
                pos += r[1]
            if call.returns:
                ret = int.from_bytes(raw[pos:pos + 8], "little", signed=name.startswith("unpack32"))
        else:
            ret = call.produce()
            ret = ret if call.returns else None
        self._state = _chain(self._state, name, call, ins, [_read(r) for r in call.outputs], ret)
        if _is_check(j, self._count):
            want = t["checks"][8 * self._check:8 * self._check + 8]
            self._check += 1
            if self._state != want:
                raise AssertionError(f"{self._key}: reference calls #{j // CHECK_EVERY * CHECK_EVERY}..#{j} (the last "
                                     f"{name}{args}): inputs or outputs differ from the reference's recorded calls")
        return ret

    def done(self):
        """Every recorded call was made, so every checkpoint was compared."""
        assert self._j == self._count, f"{self._key}: {self._j} of the {self._count} recorded reference calls were made"
