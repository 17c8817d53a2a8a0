"""Abundance vectors with the reference's interface (kmermaid/abundance.py:18-172): `kmer count -m
VEC_COUNT / VEC_COUNT_MASKED` writes, for every (record, strand), a vector holding at each k-mer's start
position the number of its occurrences (masked: in OTHER records only), one `REF___STRAND.gz` per vector
with a "# k=K" first line.

DELIBERATE FIX: the reference's AbundanceVector.add_count first calls the abstract base method, which raises
NotImplementedError (abundance.py:123 -> :60), so both modes crash as shipped (SURVEY.md Appendix A4).
The call is dropped here; everything else follows the reference, and the goldens were produced by the
reference with that one abstract method neutralised (tests/golden/golden_vec.json).

Two producers fill the same files: the host classes below (records fed one by one through
KJoiner.join_vector_count*, the reference's protocol for host batches) and the device path
(Engine.write_vectors: run lengths scattered back through the window positions by kmg_abundance_scatter in
key-range passes, the text formatted on the device; `device_vectors` returns the same vectors as arrays).
The reference's LOCAL memory mode keeps the vectors in HDF5 files while joining (abundance.py:175-303);
here LOCAL and NORMAL differ in nothing: the vectors live in device memory either way."""
from __future__ import annotations

import gzip
import os
from typing import Dict, Iterable, List, Set, Tuple

import numpy as np


def vector_text(counts: np.ndarray, k: int) -> bytes:
    """b"# k=K\\n" + one decimal per line (abundance.py:168-172), without a Python loop."""
    v = np.asarray(counts).astype(np.int64)
    nd = np.ones(v.shape, np.int64)
    t = v.copy()
    while True:
        t = t // 10
        more = t > 0
        if not more.any():
            break
        nd += more
    off = np.concatenate(([0], np.cumsum(nd + 1)))
    out = np.empty(int(off[-1]), np.uint8)
    out[off[1:] - 1] = 10
    rest = v.copy()
    for d in range(int(nd.max()) if v.size else 0):  # d-th digit from the right
        sel = nd > d
        out[off[1:][sel] - 2 - d] = 48 + rest[sel] % 10
        rest = rest // 10
    return b"# k=%d\n" % k + out.tobytes()


def vector_paths(dirpath: str, vectors: Iterable[Tuple[str, str]]) -> List[str]:
    """abundance.py:148-172: the extension is removed from `dirpath`, which must not be a file and is created
    (also when no vector follows); the path of the gz file of every (ref, strand) in `vectors`."""
    dirpath = os.path.splitext(dirpath)[0]
    if os.path.isfile(dirpath):
        raise AssertionError
    print('Writing output in "%s"' % dirpath)
    os.makedirs(dirpath, exist_ok=True)
    return [os.path.join(dirpath, "%s___%s.gz" % (ref, strand)) for ref, strand in vectors]


def check_unique_names(names: List[str]) -> None:
    if len(set(names)) != len(names):
        # two records of one name write the same vector: the reference refuses the second write
        raise AssertionError("can't update non-zero count w/o replace: records share a name")


def write_vectors(vectors: Dict[str, Dict[str, np.ndarray]], k: int, dirpath: str) -> None:
    """Host vectors to files: one gz file per (ref, strand) (see vector_paths; the device writer is
    Engine.write_vectors)."""
    keys = [(ref, strand) for ref, per in vectors.items() for strand in per]
    for (ref, strand), path in zip(keys, vector_paths(dirpath, keys)):
        with gzip.open(path, "wb") as oh:
            oh.write(vector_text(vectors[ref][strand], k))


class AbundanceVectorBase:
    _ks: Set[int] = set()

    def check_length(self, k: int) -> None:
        self._ks.add(k)
        if len(self._ks) != 1:
            raise AssertionError(f"inconsistent sequence lengths: {self._ks}")


class AbundanceVector(AbundanceVectorBase):
    """Host-side vectors (abundance.py:92-172), one instance per join."""

    def __init__(self):
        self._ks = set()  # (the reference shares these between instances: class attributes, SURVEY §8b)
        self._data: Dict[str, Dict[str, np.ndarray]] = {}

    def add_count(self, ref: str, strand: str, pos: int, count: int, k: int, replace: bool = False) -> None:
        self.check_length(k)
        self.add_ref(ref, strand, pos + 1)
        if not replace and self._data[ref][strand][pos] != 0:
            raise AssertionError(f"can't update non-zero count w/o replace: {ref},{strand},{pos},{count}")
        self._data[ref][strand][pos] = count

    def add_ref(self, ref: str, strand: str, size: int) -> None:
        per = self._data.setdefault(ref, {})
        if strand not in per:
            per[strand] = np.zeros(size, np.int64)
        elif size > per[strand].shape[0]:
            per[strand] = np.concatenate([per[strand], np.zeros(size - per[strand].shape[0], np.int64)])

    def write_to(self, dirpath: str) -> None:
        write_vectors(self._data, list(self._ks)[0] if self._ks else 0, dirpath)


AbundanceVectorLocal = AbundanceVector  # see the module docstring


def device_vectors(engine, d, k: int, rc: bool, masked: bool) -> Dict[str, Dict[str, np.ndarray]]:
    """{ref: {"+"/"-": counts}} of one DeviceInput, computed on the GPU.  A vector ends at its last
    non-zero entry (add_ref grows it only up to the positions that were written, abundance.py:137-146)."""
    names = d.flat.names
    check_unique_names(names)
    plus, minus = engine.abundance(d, k, rc, masked)
    starts = d.flat.rec_starts.astype(np.int64)
    out: Dict[str, Dict[str, np.ndarray]] = {}
    for r, name in enumerate(names):
        b, e = int(starts[r]), int(starts[r + 1]) - 1
        for label, vec in (("+", plus), ("-", minus)):
            v = vec[b:e]
            nz = np.flatnonzero(v)
            if nz.size:
                out.setdefault(name, {})[label] = v[: int(nz[-1]) + 1]
    return out
