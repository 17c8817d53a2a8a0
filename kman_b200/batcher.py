"""Batching front end with the reference's interface (kmermaid/batcher.py).

`FastaBatcher(...).do(fasta, k).collection` is the call the three `kmer` commands make
(kmermaid/scripts/kmer_count.py:100-118).  In the reference it runs the per-window Python
loop, fills batches of `size` k-mers and writes/re-sorts every batch file.  Here it parses
the FASTA on the host, moves the flat base buffer to HBM and returns ONE `DeviceBatch`;
extraction and sorting run on the GPU when the joiner (or a record view) asks for them.
`scan_mode`, `threads`, `size` and `tmp` are accepted and validated exactly as the reference
does, but cannot change results (they must not in the reference either: SURVEY.md §8a).
"""
from __future__ import annotations

import multiprocessing as mp
import os
import tempfile
from enum import Enum
from typing import Any, List, Optional, Tuple, Type, Union

from kman_b200 import alphabet as ab, fasta
from kman_b200.alphabet import NATYPES
from kman_b200.batch import Batch, DeviceBatch
from kman_b200.seq import KMer, Sequence

TMP_DIR = tempfile.TemporaryDirectory


class BatcherBase:
    """Collection of equally sized batches (kmermaid/batcher.py:27-153)."""

    DEFAULT_BATCH_SIZE = int(1e6)
    DEFAULT_NATYPE = NATYPES.DNA
    _type: Type[Sequence] = KMer

    def __init__(self, size: int, natype: Optional[NATYPES] = None, tmp: Optional[Union[TMP_DIR, str]] = None):
        self.__size = self.DEFAULT_BATCH_SIZE
        self.__natype = self.DEFAULT_NATYPE
        self.size = size
        self.natype = natype
        if isinstance(tmp, TMP_DIR):
            self._tmpH = tmp
            self._tmp = tmp.name
        elif isinstance(tmp, str):
            self._tmp = tmp
        else:
            self._tmp = tempfile.gettempdir()
        self._batches: List[Any] = [Batch.from_batcher(self.type, self.size, self.tmp)]

    @property
    def size(self) -> int:
        return self.__size

    @size.setter
    def size(self, size: Optional[int]) -> None:
        if size is not None:
            if size < 1:
                raise AssertionError
            self.__size = size

    type = property(lambda self: self._type)

    @property
    def natype(self):
        return self.__natype

    @natype.setter
    def natype(self, natype: Optional[NATYPES]) -> None:
        if natype is not None:
            if natype not in NATYPES:
                raise AssertionError
            self.__natype = natype

    collection = property(lambda self: self._batches)
    tmp = property(lambda self: self._tmp)

    def new_batch(self) -> None:
        if self.collection[-1].is_full():
            self.collection[-1].write()
            self._batches.append(Batch.from_batcher(self.type, self.size, self.tmp))

    def add_record(self, record: Any) -> None:
        self.new_batch()
        self.collection[-1].add(record)

    def write_all(self, f: str = "as_fasta", doSort: bool = False, verbose: bool = False) -> None:
        # NB the reference forwards (f, doSort) positionally into Batch.write(doSort, force)
        # (batcher.py:153 vs batch.py:281, SURVEY Appendix A3), i.e. it always sorts.
        for b in self.collection:
            if b.current_size != 0:
                b.write(True, doSort)


class BatcherThreading(BatcherBase):
    """Adds the thread clamp and the feed modes (kmermaid/batcher.py:156-288)."""

    class FEED_MODE(Enum):
        REPLACE = 1
        FLOW = 2
        APPEND = 3

    def __init__(self, size: int, threads: int = 1, natype: Optional[NATYPES] = None, tmp: Optional[str] = None):
        super().__init__(size, natype, tmp)
        self.threads = threads

    @property
    def threads(self) -> int:
        return self.__threads

    @threads.setter
    def threads(self, t: int) -> None:
        self.__threads = max(1, min(t, mp.cpu_count()))

    def feed_collection(self, new_collection: List[Any], mode: "BatcherThreading.FEED_MODE" = FEED_MODE.FLOW) -> None:
        if any(b.type != self.type for b in new_collection):
            raise AssertionError
        if mode == self.FEED_MODE.REPLACE:
            self._batches = new_collection
        elif mode == self.FEED_MODE.FLOW:
            # device batches are not re-packed into fixed-size host batches: flowing them is
            # appending them (results do not depend on batch boundaries)
            for b in list(new_collection):
                if isinstance(b, DeviceBatch):
                    self._batches.append(b)
                else:
                    for record in b.record_gen():
                        self.add_record(record)
                    b.reset()
            new_collection.clear()
        elif mode == self.FEED_MODE.APPEND:
            self._batches.extend(new_collection)

    @staticmethod
    def from_files(dirPath: str, threads: int, t: Type = KMer, isFasta: bool = True, reSort: bool = False) -> List[Batch]:
        if not os.path.isdir(dirPath):
            raise AssertionError
        return [Batch.from_file(os.path.join(dirPath, f), t, isFasta, reSort=reSort) for f in sorted(os.listdir(dirPath))]


class FastaBatcher(BatcherThreading):
    """FASTA file -> k-mer batches (kmermaid/batcher.py:291-487)."""

    class MODE(Enum):
        KMERS = 1
        RECORDS = 2

    def __init__(self, scan_mode: "FastaBatcher.MODE" = MODE.KMERS, reverse: bool = False, threads: int = 1,
                 size: int = BatcherThreading.DEFAULT_BATCH_SIZE, natype: NATYPES = BatcherThreading.DEFAULT_NATYPE,
                 tmp: str = tempfile.gettempdir(), alphabet: Optional[str] = None, canonical: bool = False):
        super().__init__(size, threads, natype, tmp)
        self.mode = scan_mode
        self.doReverseComplement = reverse
        if type(canonical) is not bool or (canonical and reverse):
            raise AssertionError("canonical is a bool and excludes reverse (canonical k-mers cover both strands)")
        self.canonical = canonical  # one k-mer per window: the smaller of it and its reverse complement
        self.alphabet = alphabet or ab.default_alphabet()

    @property
    def mode(self):
        return self._mode

    @mode.setter
    def mode(self, m) -> None:
        if m not in self.MODE:
            raise AssertionError
        self._mode = m

    @property
    def doReverseComplement(self) -> bool:
        return self._doReverseComplement

    @doReverseComplement.setter
    def doReverseComplement(self, rc) -> None:
        if type(rc) is not bool:
            raise AssertionError
        self._doReverseComplement = rc

    def do(self, fasta_path: str, k: int, feedMode: BatcherThreading.FEED_MODE = BatcherThreading.FEED_MODE.APPEND) -> "FastaBatcher":
        """Batch a FASTA file (batcher.py:454-487).  AssertionError if the file is missing or
        k <= 1; `.gz` accepted."""
        if not os.path.isfile(fasta_path):
            raise AssertionError(f"input file not found: {fasta_path}")
        if k <= 1:
            raise AssertionError(f"k must be >= 1, got {k} instead.")
        from kman_b200.engine import get_engine

        eng = get_engine()
        if os.environ.get("KMG_GPU_LOADER", "1") != "0":
            d = eng.load_fasta(fasta_path, self.alphabet, self.natype)  # text -> flat buffer on the GPU
        else:
            d = eng.upload(fasta.read_fasta(fasta_path), self.alphabet, self.natype)
        batch = DeviceBatch(eng, d, k, self.doReverseComplement, self.natype, self.tmp, self.size, self.canonical)
        self.feed_collection([batch], feedMode)
        return self


class FastaRecordBatcher(BatcherThreading):
    """One FASTA record -> k-mer batches (kmermaid/batcher.py:490-613)."""

    def __init__(self, size: int, threads: int = 1, natype: NATYPES = NATYPES.DNA, tmp: str = tempfile.gettempdir()):
        super().__init__(size=size, threads=threads, natype=natype, tmp=tmp)
        self._doReverseComplement = False
        self.alphabet = ab.default_alphabet()

    @property
    def doReverseComplement(self) -> bool:
        return self._doReverseComplement

    @doReverseComplement.setter
    def doReverseComplement(self, rc) -> None:
        if type(rc) is not bool:
            raise AssertionError
        self._doReverseComplement = rc

    def do(self, record: Tuple[str, str], k: int, verbose: bool = True) -> "FastaRecordBatcher":
        from kman_b200.engine import get_engine

        eng = get_engine()
        d = eng.upload(fasta.from_records([record]), self.alphabet, self.natype)
        self.feed_collection(
            [DeviceBatch(eng, d, k, self.doReverseComplement, self.natype, self.tmp, self.size)], self.FEED_MODE.APPEND)
        return self

    @staticmethod
    def from_parent(parent: "FastaBatcher") -> "FastaRecordBatcher":
        b = FastaRecordBatcher(parent.size, parent.threads, parent.natype, parent.tmp)
        b._doReverseComplement = parent.doReverseComplement
        b.alphabet = getattr(parent, "alphabet", b.alphabet)
        return b


def load_batches(previous_batches: str, threads: int = 1, re_sort: bool = False, natype: NATYPES = NATYPES.DNA,
                 alphabet: Optional[str] = None) -> List:
    """Previously generated batch files (`kmer batch` output, plain or .gz) re-imported as device keys
    (kmermaid/batcher.py:616-636).

    DELIBERATE FIX: the reference's guard is inverted -- `len(os.listdir(dir)) > 0` raises, so as shipped it
    rejects every folder that holds batches (batcher.py:631, SURVEY.md Appendix A5) and `-B` can never
    work.  Here the folder must exist and hold at least one file, as the reference's own docstring says
    ("input folder must exist and be non-empty").  `re_sort` is accepted and irrelevant: the device path
    always sorts."""
    if not os.path.isdir(previous_batches) or len(os.listdir(previous_batches)) == 0:
        raise AssertionError(f"folder with previous batches empty or not found: {previous_batches}")
    from kman_b200.batch import LoadedKmerBatch
    from kman_b200.engine import get_engine

    paths = [os.path.join(previous_batches, f) for f in sorted(os.listdir(previous_batches))]
    paths = [p for p in paths if os.path.isfile(p)]
    if not paths:
        raise AssertionError(f"folder with previous batches empty or not found: {previous_batches}")
    return [LoadedKmerBatch(get_engine(), paths, natype, tempfile.gettempdir(), alphabet)]
