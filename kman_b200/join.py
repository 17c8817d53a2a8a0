"""Joining front end with the reference's interface (kmermaid/join.py).

`KJoinerThreading(mode, memory).join(batches, outpath)` is the call the `kmer count` / `kmer
uniq` commands make.  In the reference it is an n-way `heapq.merge` over every batch file
plus a grouping loop (join.py:63-130).  Here, for `DeviceBatch` inputs, it is the GPU path:
extract -> radix sort -> run-length (count) or singleton selection (uniq) -> text emission,
in key-range passes when the input does not fit the device at once, streamed to the output
file in chunks.  The emitted bytes equal the reference's
(join.py:262 ">%s\\n%s\\n", join.py:284 "%s\\t%d\\n"); an empty result leaves an empty file.
A SEQ_COUNT join can keep only the lines whose count is in `count_range` (`kmer count --min-count /
--max-count`): the same file with the other lines removed, on every path.
"""
from __future__ import annotations

import logging
import multiprocessing as mp
from enum import Enum
from typing import IO, Any, Iterator, List, Optional, Tuple

import numpy as np

from kman_b200 import fasta
from kman_b200.batch import Batch, BatchAppendable, DeviceBatch
from kman_b200.seq import SequenceCoords


class Crawler:
    """Record-level view over batches (kmermaid/join.py:36-130); used for host batches and for
    callers that want the reference's iterator protocol.  The GPU join does not go through it."""

    doSort = False
    doSmart = False
    verbose = True
    desc = ""

    @staticmethod
    def count_records(batches: List[Any]) -> int:
        return sum(b.current_size for b in batches)

    def do_records(self, batches: List[Any]) -> Iterator[Tuple[str, str]]:
        from heapq import merge

        if any(type(b) not in (Batch, BatchAppendable, DeviceBatch) for b in batches):
            raise AssertionError()
        gens = [((str(r.header), str(r.seq)) for r in (b.sorted(self.doSmart) if self.doSort or isinstance(b, DeviceBatch)
                                                       else b.record_gen(self.doSmart))) for b in batches]
        yield from merge(*gens, key=lambda x: x[1])

    def do_batch(self, batches: List[Any]) -> Iterator[Tuple[List[str], str]]:
        cur_seq, headers = None, []
        for header, seq in self.do_records(batches):
            if cur_seq is None:
                cur_seq, headers = seq, [header]
            elif seq == cur_seq:
                headers.append(header)
            else:
                yield headers, cur_seq
                cur_seq, headers = seq, [header]
        if cur_seq is None:
            logging.error("nothing to crawl")
            return
        yield headers, cur_seq


class KJoiner:
    """K-way joining (kmermaid/join.py:133-391)."""

    class MODE(Enum):
        UNIQUE = 1
        SEQ_COUNT = 2
        VEC_COUNT = 3
        VEC_COUNT_MASKED = 4

    class MEMORY(Enum):
        NORMAL = 1
        LOCAL = 2

    DEFAULT_MODE = MODE.UNIQUE
    DEFAULT_MEMORY = MEMORY.NORMAL

    def __init__(self, mode: Optional["KJoiner.MODE"] = None, memory: Optional["KJoiner.MEMORY"] = None):
        self.__mode = self.DEFAULT_MODE
        self.__memory = self.DEFAULT_MEMORY
        self.__count_range: Tuple[int, Optional[int]] = (1, None)
        if mode is not None:
            self.mode = mode
        if memory is not None:
            self.memory = memory

    @property
    def mode(self):
        return self.__mode

    @mode.setter
    def mode(self, mode) -> None:
        if mode not in self.MODE:
            raise AssertionError
        self.__mode = mode

    @property
    def memory(self):
        return self.__memory

    @memory.setter
    def memory(self, memory) -> None:
        if memory not in self.MEMORY:
            raise AssertionError
        self.__memory = memory

    @property
    def count_range(self) -> Tuple[int, Optional[int]]:
        """(min_count, max_count) of the SEQ_COUNT lines written; max_count None: no upper limit."""
        return self.__count_range

    @count_range.setter
    def count_range(self, r: Tuple[int, Optional[int]]) -> None:
        lo, hi = int(r[0]), None if r[1] is None else int(r[1])
        self._check_range(lo, hi)
        self.__count_range = (lo, hi)

    def _check_range(self, lo: int, hi: Optional[int]) -> Optional[Tuple[int, int]]:
        """(min_count, max_count) for the native calls, None for every line; AssertionError for a bad range or a
        range outside SEQ_COUNT."""
        if (lo, hi) == (1, None):  # (the default: no engine import on the host path)
            return None
        from kman_b200.engine import count_range

        rng = count_range(lo, hi)
        if rng is not None and self.mode != self.MODE.SEQ_COUNT:
            raise AssertionError(f"--min-count / --max-count apply to SEQ_COUNT only, not to {self.mode.name}")
        return rng

    @property
    def join_function(self):
        return {
            self.MODE.UNIQUE: self.join_unique,
            self.MODE.SEQ_COUNT: self.join_sequence_count,
            self.MODE.VEC_COUNT: self.join_vector_count,
            self.MODE.VEC_COUNT_MASKED: self.join_vector_count_masked,
        }[self.mode]

    @staticmethod
    def join_unique(headers: List[str], seq: str, OH: IO, **kwargs) -> Optional[Tuple[str, str]]:
        if len(headers) != 1:
            return None
        OH.write(">%s\n%s\n" % (headers[0], seq))
        return (headers[0], seq)

    @staticmethod
    def join_sequence_count(headers: List[str], seq: str, OH: IO, **kwargs) -> Tuple[str, int]:
        OH.write("%s\t%d\n" % (seq, len(headers)))
        return (seq, len(headers))

    @staticmethod
    def join_vector_count(headers: List[str], seq: str, OH, vector=None, **kwargs) -> None:
        """join.py:287-308: every member of the group stores the group's size at its start position."""
        hcount = len(headers)
        for header in headers:
            c = SequenceCoords.from_str(header)
            vector.add_count(c.ref, c.strand.label, int(c.start), hcount, len(seq))

    @staticmethod
    def join_vector_count_masked(headers: List[str], seq: str, OH, vector=None, **kwargs) -> None:
        """join.py:310-335: only groups spread over several records count, and only the other records' members."""
        coords = [SequenceCoords.from_str(h) for h in headers]
        if len(coords) != 1 and len({c.ref for c in coords}) != 1:
            for c in coords:
                vector.add_count(c.ref, c.strand.label, int(c.start), sum(1 for o in coords if o.ref != c.ref), len(seq))

    # ---- GPU join ------------------------------------------------------------------------------
    @staticmethod
    def _merged_device_input(batches: List[DeviceBatch]):
        """One DeviceInput covering every batch (several FASTA files appended: their records are
        concatenated in batch order, which is the order heapq.merge breaks ties in)."""
        if len(batches) == 1:
            return batches[0].device_input
        b0 = batches[0]
        if any((b.k, b.reverse, b.canonical, b.natype, b.device_input.alphabet)
               != (b0.k, b0.reverse, b0.canonical, b0.natype, b0.device_input.alphabet) for b in batches):
            raise AssertionError("batches were built with different k / reverse / canonical / alphabet settings")
        flats = [b.device_input.flat for b in batches]
        bases = np.concatenate([f.bases for f in flats])
        starts, names, titles, off = [], [], [], 0
        for f in flats:
            starts.append(f.rec_starts[:-1].astype(np.uint64) + np.uint64(off))
            names += f.names
            titles += f.titles
            off += int(f.bases.shape[0])
        starts.append(np.array([off], np.uint64))
        flat = fasta.FlatInput(bases, np.concatenate(starts), names, titles)
        return b0._eng.upload(flat, b0.device_input.alphabet, b0.natype)

    def _join_device(self, batches: List[DeviceBatch], outpath: str) -> None:
        b0 = batches[0]
        if self.mode.name.startswith("VEC_"):
            from kman_b200.batch import LoadedKmerBatch

            if any(isinstance(b, LoadedKmerBatch) for b in batches):
                raise AssertionError("abundance vectors need the FASTA input, not re-imported batch files")
            if any(b.canonical for b in batches):
                raise AssertionError("abundance vectors are per strand: not with canonical k-mers")
            d = self._merged_device_input(batches)
            # join.py:370-372 -> abundance.py:148-172, in key-range passes with device text (KMG_DEVICE_BUDGET applies)
            b0._eng.write_vectors(d, b0.k, b0.reverse, self.mode == self.MODE.VEC_COUNT_MASKED, outpath)
            return
        from kman_b200.batch import LoadedKmerBatch

        lo, hi = self._check_range(*self.count_range) or (1, None)
        if any(isinstance(b, LoadedKmerBatch) for b in batches):
            # `-B`: re-imported batch files carry their own headers (one LoadedKmerBatch covers a folder)
            if len(batches) != 1:
                raise AssertionError("re-imported batch files cannot be joined together with other batches")
            with open(outpath, "wb") as oh:
                if self.mode == self.MODE.SEQ_COUNT:
                    b0._eng.write_count(b0.device_input, b0.k, False, oh, min_count=lo, max_count=hi)
                else:
                    oh.write(b0.uniq_text())
            return
        d = self._merged_device_input(batches)
        rc = b0.strand_rule  # (engine.CANONICAL for --canonical batches)
        # key-range passes and chunked text: device memory is bounded by the largest pass, host memory by a
        # text chunk (KMG_DEVICE_BUDGET overrides the device budget)
        with open(outpath, "wb") as oh:  # join.py:351 opens "w+": the file exists even when empty
            if self.mode == self.MODE.SEQ_COUNT:
                b0._eng.write_count(d, b0.k, rc, oh, min_count=lo, max_count=hi)
            else:
                b0._eng.write_uniq(d, b0.k, rc, oh)

    def join(self, batches: List[Any], outpath: str) -> None:
        rng = self._check_range(*self.count_range)
        live = [b for b in batches if b is not None and not (isinstance(b, Batch) and b.current_size == 0)]
        if live and all(isinstance(b, DeviceBatch) for b in live):
            print("Joining...")
            return self._join_device(live, outpath)
        if any(isinstance(b, DeviceBatch) for b in live):
            raise AssertionError("cannot join device batches together with host batches")
        # host batches only (records built by callers through the Batch API): reference protocol
        print("Joining...")
        if self.mode.name.startswith("VEC_"):  # join.py:337-372
            from kman_b200.abundance import AbundanceVector

            vector = AbundanceVector()
            for headers, seq in Crawler().do_batch(live):
                self.join_function(headers, seq, OH=outpath, vector=vector)
            vector.write_to(outpath)
            return
        with open(outpath, "w+") as oh:
            for headers, seq in Crawler().do_batch(live):
                if rng is None or rng[0] <= len(headers) <= rng[1]:
                    self.join_function(headers, seq, OH=oh)


class KJoinerThreading(KJoiner):
    """Adds the thread / batch-size knobs of kmermaid/join.py:394-480.  They are validated the
    same way and do not change results (the reference's threaded join is defective, SURVEY
    Appendix A1; results here always equal its 1-thread output)."""

    def __init__(self, mode=None, memory=None):
        super().__init__(mode, memory)
        self._threads = 1
        self.__batch_size = 10
        self.__doSort = False

    @property
    def doSort(self) -> bool:
        return self.__doSort

    @doSort.setter
    def doSort(self, v) -> None:
        if type(v) is not bool:
            raise AssertionError
        self.__doSort = v

    @property
    def threads(self) -> int:
        return self._threads

    @threads.setter
    def threads(self, t: int) -> None:
        self._threads = max(1, min(t, mp.cpu_count()))

    @property
    def batch_size(self) -> int:
        return self.__batch_size

    @batch_size.setter
    def batch_size(self, n) -> None:
        if type(n) is not int or n < 2:
            raise AssertionError
        self.__batch_size = n
