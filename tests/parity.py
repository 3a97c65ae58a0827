"""Comparison helpers shared by the parity tests and tools/gpu_parity_report.py."""
from __future__ import annotations

import hashlib

import numpy as np

from instance_stixels_b200 import _lib as L


def column_lengths(sections: np.ndarray) -> np.ndarray:
    """Number of stixels per column of a [C][200] Section array (type == -1 terminates)."""
    term = sections["type"] == -1
    has = term.any(axis=1)
    n = np.where(has, term.argmax(axis=1), sections.shape[1])
    return n


def compare_sections(ours: np.ndarray, ref: np.ndarray, rtol: float = 1e-4) -> dict:
    """Column-by-column comparison of two [C][200] Section arrays.

    exact   : same number of stixels and identical type / vB / vT / class in every stixel
    bitwise : additionally bit-identical disparity, cost and instance means
    close   : additionally float fields within `rtol` relative
    """
    C = ours.shape[0]
    n_o, n_r = column_lengths(ours), column_lengths(ref)
    exact = np.zeros(C, bool)
    bitwise = np.zeros(C, bool)
    close = np.zeros(C, bool)
    max_rel = {"disparity": 0.0, "cost": 0.0, "instance_meanx": 0.0, "instance_meany": 0.0}
    first_bad = []
    for c in range(C):
        if n_o[c] != n_r[c]:
            if len(first_bad) < 8:
                first_bad.append((c, "count", int(n_o[c]), int(n_r[c])))
            continue
        a, b = ours[c, :n_o[c]], ref[c, :n_r[c]]
        ok = all(np.array_equal(a[f], b[f]) for f in ("type", "vB", "vT", "semantic_class"))
        exact[c] = ok
        if not ok:
            if len(first_bad) < 8:
                j = int(np.argmax([(a[k]["type"], a[k]["vB"], a[k]["vT"], a[k]["semantic_class"]) !=
                                   (b[k]["type"], b[k]["vB"], b[k]["vT"], b[k]["semantic_class"])
                                   for k in range(len(a))]))
                first_bad.append((c, "struct", j, a[j].tolist(), b[j].tolist()))
            continue
        bw, cl = True, True
        for f in max_rel:
            x, y = a[f], b[f]
            if not np.array_equal(x.view(np.int32), y.view(np.int32)):
                bw = False
            with np.errstate(invalid="ignore", divide="ignore"):
                rel = np.abs(x - y) / np.maximum(np.abs(y), 1e-6)
            rel = np.where(np.isfinite(rel), rel, 0.0)
            if rel.size:
                max_rel[f] = max(max_rel[f], float(rel.max()))
                if rel.max() > rtol:
                    cl = False
        bitwise[c] = bw
        close[c] = cl
    return dict(columns=C, exact=float(exact.mean()), bitwise=float(bitwise.mean()), close=float(close.mean()),
                max_rel=max_rel, first_bad=first_bad, stixels_ours=int(n_o.sum()), stixels_ref=int(n_r.sum()))


def same_used_sections(a: np.ndarray, b: np.ndarray) -> bool:
    """Byte equality of the USED part of two [C][200] Section arrays: per column the stixels and the
    type == -1 terminator.  Entries after the terminator are never written (like the reference's
    d_stixels, StixelsKernels.cu:951-955) and hold whatever an earlier frame left there."""
    na, nb = column_lengths(a), column_lengths(b)
    if not np.array_equal(na, nb):
        return False
    used = np.arange(a.shape[1])[None, :] <= na[:, None]
    return bool(np.array_equal(a[used].view(np.uint8), b[used].view(np.uint8)))


def partition_of(instances: np.ndarray) -> dict:
    """{(class, label): frozenset of (column, index)} ignoring noise; plus the noise set under key None."""
    groups: dict = {}
    for r in instances:
        key = None if r["label"] < 0 else (int(r["semantic_class"]), int(r["label"]))
        groups.setdefault(key, set()).add((int(r["column"]), int(r["index"])))
    return groups


def compare_instances(ours: np.ndarray, ref: np.ndarray) -> dict:
    """Instance ids are compared up to label permutation (per class)."""
    po, pr = partition_of(ours), partition_of(ref)
    so = {frozenset(v) for k, v in po.items() if k is not None}
    sr = {frozenset(v) for k, v in pr.items() if k is not None}
    keys_o = {(int(r["column"]), int(r["index"])) for r in ours}
    keys_r = {(int(r["column"]), int(r["index"])) for r in ref}
    return dict(n_ours=len(ours), n_ref=len(ref), same_keys=keys_o == keys_r, clusters_ours=len(so),
                clusters_ref=len(sr), same_partition=(so == sr and po.get(None, set()) == pr.get(None, set())))


def sections_digest(sections: np.ndarray) -> str:
    """SHA-256 of the column lengths and the stixels of a [C][200] Section array: equal digests mean identical
    boundaries, types and classes and bit-identical floats on every column (the terminators are not included)."""
    n = column_lengths(sections)
    used = np.arange(sections.shape[1])[None, :] < n[:, None]
    h = hashlib.sha256(n.astype(np.int32).tobytes())
    h.update(np.ascontiguousarray(sections[used]).tobytes())
    return h.hexdigest()


def partition_digest(instances: np.ndarray) -> str:
    """SHA-256 of the instance stixels and their partition up to label permutation: equal digests mean what
    compare_instances calls same_keys and same_partition."""
    groups = partition_of(instances)
    keys = sorted((int(r["column"]), int(r["index"])) for r in instances)
    clusters = sorted(sorted(v) for k, v in groups.items() if k is not None)
    noise = sorted(groups.get(None, ()))
    return hashlib.sha256(repr((keys, clusters, noise)).encode()).hexdigest()


def array_digest(a: np.ndarray) -> str:
    """SHA-256 of the bytes of an array (bit-exact comparison of a stored table)."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def bit_equal(a: np.ndarray, b: np.ndarray) -> float:
    """Fraction of bit-identical float32 elements."""
    return float((a.view(np.int32) == b.view(np.int32)).mean())


SECTION_DTYPE = L.SECTION_DTYPE
