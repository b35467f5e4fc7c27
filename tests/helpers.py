"""Shared helpers for the parity tests: compare a GPU result block with the oracle's."""
import math
import struct

import numpy as np

from databend_b200 import abi
from databend_b200.block import Column, DataBlock


def sorted_group_result_from_block(block: DataBlock, n_aggs: int, n_keys: int):
    """GPU result block [aggs..., keys...] -> dict sorted by key (assert_block_value_sort_eq)."""
    keys = [block.columns[n_aggs + k] for k in range(n_keys)]
    order = np.arange(block.num_rows)
    if n_keys:
        kv = keys[0].values().astype(np.int64) if keys[0].dtype != abi.U64 else keys[0].values().view(np.int64)
        kvalid = keys[0].valid_mask()
        order = np.lexsort((kv, ~kvalid))  # valid keys ascending, then NULL key last
    out = {"keys": [], "key_valid": [], "aggs": [], "agg_valid": []}
    for k in keys:
        out["keys"].append(k.values()[order])
        out["key_valid"].append(k.valid_mask()[order])
    for a in range(n_aggs):
        c = block.columns[a]
        out["aggs"].append(c.values()[order])
        out["agg_valid"].append(c.valid_mask()[order])
    return out


def sorted_group_result_from_oracle(res, key_dtypes):
    keys, kvalid, aggs, avalid, adt = res
    n = len(aggs[0]) if aggs else (len(keys[0]) if keys else 0)
    order = np.arange(n)
    typed_keys = []
    for k, dt in zip(keys, key_dtypes):
        from databend_b200.block import np_dtype
        nd = np_dtype(dt)
        typed_keys.append(k.astype(np.uint64).view(np.uint64).astype(nd) if nd.itemsize < 8 else k.view(nd))
    if keys:
        kv = typed_keys[0].astype(np.int64) if key_dtypes[0] != abi.U64 else typed_keys[0].view(np.int64)
        order = np.lexsort((kv, ~kvalid[0]))
    out = {"keys": [k[order] for k in typed_keys], "key_valid": [v[order] for v in kvalid],
           "aggs": [a[order] for a in aggs], "agg_valid": [v[order] for v in avalid]}
    return out


def assert_group_results_equal(gpu, orc, float_exact=True, rtol=0.0):
    assert len(gpu["aggs"]) == len(orc["aggs"])
    for k in range(len(gpu["keys"])):
        np.testing.assert_array_equal(gpu["key_valid"][k], orc["key_valid"][k])
        m = orc["key_valid"][k]
        np.testing.assert_array_equal(gpu["keys"][k][m], orc["keys"][k][m])
    for a in range(len(gpu["aggs"])):
        np.testing.assert_array_equal(gpu["agg_valid"][a], orc["agg_valid"][a], err_msg=f"agg {a} validity")
        m = orc["agg_valid"][a]
        g, o = gpu["aggs"][a][m], orc["aggs"][a][m]
        assert g.dtype == o.dtype, (a, g.dtype, o.dtype)
        if g.dtype.kind == "f" and not float_exact:
            np.testing.assert_allclose(g, o, rtol=rtol, atol=0)
        elif g.dtype.kind == "f":
            np.testing.assert_array_equal(g.view(np.uint64 if g.itemsize == 8 else np.uint32),
                                          o.view(np.uint64 if o.itemsize == 8 else np.uint32), err_msg=f"agg {a}")
        else:
            np.testing.assert_array_equal(g, o, err_msg=f"agg {a}")


def derive_join_rows(kind: str, probe_key, build_key, pairs):
    """Expected output row indices of a probe-side ("left") join from the oracle's INNER pairs
    (probe_idx, build_idx): the same derivation the GPU join tests use.
      inner -> the pairs;  left -> pairs + (p, None) for unmatched probe rows;
      semi  -> probe rows with a match, once;  anti -> probe rows without a match (NULL keys too)."""
    pi, bi = pairs
    n = len(probe_key)
    matched = np.zeros(n, dtype=bool)
    matched[pi] = True
    if kind == "inner":
        return [(int(p), int(b)) for p, b in zip(pi, bi)]
    if kind == "left":
        return [(int(p), int(b)) for p, b in zip(pi, bi)] + [(int(p), None) for p in np.nonzero(~matched)[0]]
    if kind == "semi":
        return [(int(p), None) for p in np.nonzero(matched)[0]]
    if kind == "anti":
        return [(int(p), None) for p in np.nonzero(~matched)[0]]
    raise ValueError(kind)


INT_TYPES = ["I8", "I16", "I32", "I64", "U8", "U16", "U32", "U64"]


def int_type_range(t: str):
    bits = int(t[1:])
    return (-(1 << (bits - 1)), (1 << (bits - 1)) - 1) if t[0] == "I" else (0, (1 << bits) - 1)


def float_int_boundaries(t: str, ftype: str):
    """Values of float type `ftype` ("F32" / "F64") where a rounding float -> integer cast to `t` can go
    wrong: MIN - 1, MIN - 0.5, MIN, MAX, MAX + 0.5, MAX + 1 (each to the nearest value of `ftype`) and
    both of their neighbours (so MIN - 0.49999999999999994, nextafter(2^63, 0), nextafter(-2^63, -inf),
    nextafter(2^64, 0) and the like), 2^63 and 2^64, odd integers in [2^52, 2^53), +-0, +-0.5, the
    subnormals, +-inf and NaN.  Sorted, duplicates removed, as Python floats."""
    from fractions import Fraction
    ft = np.float32 if ftype == "F32" else np.float64
    lo, hi = int_type_range(t)
    anchors = [Fraction(lo) - 1, Fraction(lo) - Fraction(1, 2), Fraction(lo), Fraction(hi), Fraction(hi) + Fraction(1, 2),
               Fraction(hi) + 1, Fraction(2) ** 63, -Fraction(2) ** 63, Fraction(2) ** 64, Fraction(1, 2), -Fraction(1, 2)]
    vals = []
    with np.errstate(over="ignore"):
        for a in anchors:
            x = ft(float(a))  # only needs to land next to the anchor
            vals += [np.nextafter(x, ft(-np.inf)), x, np.nextafter(x, ft(np.inf))]
    tiny = np.finfo(ft).smallest_subnormal
    vals += [0.0, -0.0, tiny, -tiny, np.finfo(ft).tiny, np.inf, -np.inf, 2.0 ** 52 + 1, 2.0 ** 52 + 3, -(2.0 ** 52 + 1), 1.5, -1.5, 2.5, -2.5]
    by_bits = {struct.pack("<d", float(ft(v))): float(ft(v)) for v in vals}  # keeps -0.0 apart from 0.0
    return sorted(by_bits.values(), key=lambda v: (v, math.copysign(1.0, v))) + [float("nan")]
