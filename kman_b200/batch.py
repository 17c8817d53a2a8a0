"""Batch containers with the reference's interface (kmermaid/batch.py).

`Batch` is the host-side fixed-capacity record container the reference's callers know
(in memory or backed by a temporary FASTA/TSV file, kmermaid/batch.py:19-395).
`DeviceBatch` is what the B200 path produces instead of thousands of on-disk batch files:
ONE batch whose records live in HBM as packed keys.  It offers the same duck-type the
reference's callers use (`current_size`, `type`, `tmp`, `record_gen`, `sorted`, `write`,
`unwrite`, `reset`, `is_written`, `is_full`), so `io.copy_batches` and `Crawler` accept it,
while `KJoiner.join` recognises it and stays on the GPU.
"""
from __future__ import annotations

import gzip
import os
import tempfile
import time
from typing import IO, Any, Iterator, List, Optional, Type

import numpy as np

from kman_b200.alphabet import NATYPES
from kman_b200.seq import KMer, SequenceCoords, decode_keys


def _simple_fasta(handle: IO) -> Iterator[tuple]:
    """(title, sequence) pairs of a FASTA handle, Bio.SeqIO.FastaIO.SimpleFastaParser semantics
    (the parser the reference's Batch uses, kmermaid/batch.py:13,181)."""
    title, chunks = None, []
    for line in handle:
        if line.startswith(">"):
            if title is not None:
                yield title, "".join(chunks).replace(" ", "").replace("\r", "")
            title, chunks = line[1:].rstrip(), []
        elif title is not None:
            chunks.append(line.rstrip())
    if title is not None:
        yield title, "".join(chunks).replace(" ", "").replace("\r", "")


class Batch:
    """Host record container (kmermaid/batch.py:19-395): cannot be resized; records are read
    back from the temporary file once written."""

    _fread = "from_file"
    _fwrite = "as_fasta"
    _keyAttr = "seq"
    isFasta = True
    suffix = ".fa"

    def __init__(self, t: Type, tmpDir: str, size: int = 1):
        if size < 1:
            raise AssertionError
        self.__size = int(size)
        self._remaining = self.__size
        self.__type = t
        self._tmp_dir = tmpDir
        self._tmp: Optional[str] = None
        self._written = False
        self._i = 0
        self.__records: List[Any] = [None] * self.__size

    is_written = property(lambda self: self._written)
    current_size = property(lambda self: self._i)
    size = property(lambda self: self.__size)
    remaining = property(lambda self: self._remaining)
    type = property(lambda self: self.__type)

    @property
    def collection(self):
        return None if self.__records is None else self.__records.copy()

    @property
    def tmp(self) -> str:
        if self._tmp is None:
            with tempfile.NamedTemporaryFile(mode="w+", dir=self._tmp_dir, prefix=str(hash(time.time())),
                                             suffix=self.suffix) as th:
                self._tmp = th.name
        return self._tmp

    @property
    def info(self) -> str:
        return "%s\ntype: %s\nsize: %d\ni: %d\nremaining: %d\nwritten: %r\n" % (
            self.tmp, self.type, self.size, self.current_size, self.remaining, self.is_written)

    def _checked_attr(self, name):
        if not isinstance(name, str) or not hasattr(self.type, name):
            raise AssertionError
        return name

    keyAttr = property(lambda self: self._keyAttr, lambda self, v: setattr(self, "_keyAttr", self._checked_attr(v)))
    fread = property(lambda self: self._fread, lambda self, v: setattr(self, "_fread", self._checked_attr(v)))
    fwrite = property(lambda self: self._fwrite, lambda self, v: setattr(self, "_fwrite", self._checked_attr(v)))

    def sorted(self, smart: bool = False) -> Any:
        """Stable sort by the key attribute (batch.py:156-168)."""
        if self.isFasta:
            return sorted(self.record_gen(smart), key=lambda r: getattr(r, self.keyAttr))
        return sorted(self.record_gen(smart))

    def _record_gen_from_file(self, smart: bool = False) -> Iterator[Any]:
        opener = gzip.open if self.tmp.endswith(".gz") else open
        with opener(self.tmp, "rt") as th:
            make = getattr(self.type, self.fread)
            if self.isFasta:
                for rec in _simple_fasta(th):
                    yield make(rec)
            else:
                for line in th:
                    yield make(line)

    def record_gen(self, smart: bool = False) -> Iterator[Any]:
        if self.is_written:
            yield from self._record_gen_from_file(smart)
        else:
            for r in self.__records:
                if r is not None:
                    yield r

    def check_record(self, record: Any) -> None:
        if type(record) != self.type:
            raise AssertionError(f"record must be {self.type}, not {type(record)}.")

    def add(self, record: Any) -> None:
        if self.is_full():
            raise AssertionError("this batch is full.")
        if self.is_written:
            raise AssertionError("this batch has been stored locally.")
        self.check_record(record)
        self.__records[self._i] = record
        self._i += 1
        self._remaining -= 1

    def add_all(self, recordGen) -> None:
        for r in recordGen:
            self.add(r)

    def to_write(self, doSort: bool = False) -> List[Any]:
        src = self.sorted() if doSort else self.record_gen()
        return [getattr(r, self.fwrite)() for r in src if r is not None]

    def write(self, doSort: bool = False, force: bool = False) -> None:
        if not self.is_written or force:
            out = [x if x.endswith("\n") else x + "\n" for x in self.to_write(doSort)]
            with open(self.tmp, "w+") as th:
                th.write("".join(out))
            self.__records = [None]
            self._written = True

    @staticmethod
    def from_file(path: str, t: Type = KMer, isFasta: bool = True, smart: bool = False, reSort: bool = False) -> "Batch":
        opener = gzip.open if path.endswith(".gz") else open
        with opener(path, "rt") as fh:
            n = sum(1 for _ in _simple_fasta(fh)) if isFasta else sum(1 for _ in fh)
        size = max(2, n)
        b = Batch(t, os.path.dirname(path), size)
        b._tmp = path
        b._i = size
        b._remaining = 0
        b._written = True
        b.isFasta = isFasta
        if reSort:
            b.write(doSort=True, force=True)
        return b

    @staticmethod
    def from_batcher(batch_type: Type, size: int = 1, tmp: str = tempfile.gettempdir()) -> "Batch":
        if size < 1:
            raise AssertionError(f"size cannot be 0 or negative: {size}")
        return Batch(batch_type, tmp, size)

    def reset(self) -> None:
        if self.is_written:
            os.remove(self.tmp)
        self._written = False
        self._i = 0
        self._remaining = self.size
        self.__records = [None] * self.size

    def is_full(self) -> bool:
        return self.remaining == 0

    def unwrite(self) -> None:
        if not self.is_full() and self.is_written:
            recs = list(self.record_gen())
            self.__records = [None] * self.size
            self.__records[: len(recs)] = recs
            self._written = False
            os.remove(self.tmp)


class BatchAppendable(Batch):
    """Batch that appends records straight to its file (kmermaid/batch.py:398-566); used by the
    reference only for intermediate joins."""

    def __init__(self, t: Type, tmpDir: str, size: int = 1):
        super().__init__(t, tmpDir, size)
        self._written = True
        self.isFasta = False
        self._fwrite = "as_text" if hasattr(t, "as_text") else self._fwrite

    def add(self, record: Any) -> None:
        if self.is_full():
            raise AssertionError("this batch is full.")
        self.check_record(record)
        text = getattr(record, self.fwrite)()
        with open(self.tmp, "a+") as th:
            th.write(text if text.endswith("\n") else text + "\n")
        self._i += 1
        self._remaining -= 1

    def record_gen(self, smart: bool = False) -> Iterator[Any]:
        if self._i:
            yield from self._record_gen_from_file(smart)

    def write(self, doSort: bool = False, force: bool = False) -> None:
        if doSort and self._i:
            out = [getattr(r, self.fwrite)() for r in self.sorted()]
            with open(self.tmp, "w+") as th:
                th.write("".join(x if x.endswith("\n") else x + "\n" for x in out))

    def unwrite(self) -> None:  # records only ever live in the file
        return None

    def reset(self) -> None:
        if self._i and os.path.isfile(self.tmp):
            os.remove(self.tmp)
        self._i = 0
        self._remaining = self.size


class DeviceBatch:
    """All k-mers of one FASTA input, resident on the GPU.

    Holds the flat base buffer in HBM plus (k, reverse, canonical, alphabet).  Extraction and sorting are
    run lazily by whoever needs them: `KJoiner.join` asks for key-only sorted streams in count
    mode and for keys + coordinates in uniq mode; `record_gen` / `sorted` / `write` decode
    records for callers that want the reference's record view.  `canonical`: one k-mer per window, the
    smaller of it and its reverse complement (`--canonical`; never together with `reverse`)."""

    isFasta = True
    suffix = ".fa"

    def __init__(self, engine, device_input, k: int, reverse: bool, natype: NATYPES, tmp_dir: str,
                 size: int = 1_000_000, canonical: bool = False):
        if canonical and reverse:
            raise AssertionError("canonical k-mers already cover both strands: not together with reverse")
        self._eng = engine
        self.device_input = device_input
        self.k = k
        self.reverse = reverse
        self.canonical = canonical
        self.natype = natype
        self._tmp_dir = tmp_dir
        self._size = int(size)
        self._tmp: Optional[str] = None
        self._written = False
        self._n: Optional[int] = None

    type = property(lambda self: KMer)
    size = property(lambda self: max(self._size, self.current_size))

    @property
    def strand_rule(self):
        """The engine's `rc` for this batch: engine.CANONICAL, or `reverse`."""
        if self.canonical:
            from kman_b200.engine import CANONICAL

            return CANONICAL
        return self.reverse
    remaining = property(lambda self: 0)
    is_written = property(lambda self: self._written)

    @property
    def current_size(self) -> int:
        """Number of k-mer records (valid windows, x2 with reverse complement; one per window when canonical)."""
        if self._n is None:
            from kman_b200.engine import keys_per_window

            rc = self.strand_rule
            n, n_other = self._eng.count_windows(self.device_input, self.k, rc)
            self._n = n + n_other * keys_per_window(rc)
        return self._n

    @property
    def tmp(self) -> str:
        if self._tmp is None:
            with tempfile.NamedTemporaryFile(mode="w+", dir=self._tmp_dir, prefix=str(hash(time.time())),
                                             suffix=self.suffix) as th:
                self._tmp = th.name
        return self._tmp

    def is_full(self) -> bool:
        return True

    # ---- record views (decode on the host; order as the reference's) -------------------------
    def _records(self, do_sort: bool) -> Iterator[KMer]:
        d = self.device_input
        flat = d.flat
        streams = []
        for wide in (False, True):
            a = self._eng.extract(d, self.k, self.strand_rule, wide=wide, val_bytes=8)
            if wide is False and a.n_other == 0:
                streams.append(a)
                break
            streams.append(a)
        vals = np.concatenate([s.vals_host() for s in streams])
        txt = np.concatenate([decode_keys(s.keys_host(), self.k, s.wide, self.natype) for s in streams])
        order = np.argsort(vals, kind="stable")  # emission order: position, '+' before '-'
        if do_sort:
            view = np.ascontiguousarray(txt[order]).view("S%d" % self.k).reshape(-1)
            order = order[np.argsort(view, kind="stable")]  # batch.py:156-168: stable by sequence
        starts = flat.rec_starts.astype(np.int64)
        for i in order:
            pos, minus = int(vals[i] >> np.uint64(1)), int(vals[i] & np.uint64(1))
            rec = int(np.searchsorted(starts, pos, side="right") - 1)
            st = pos - int(starts[rec])
            strand = SequenceCoords.STRAND.MINUS if minus else SequenceCoords.STRAND.PLUS
            yield KMer(flat.names[rec], st, st + self.k, txt[i].tobytes().decode("latin-1"), self.natype, strand)

    def record_gen(self, smart: bool = False) -> Iterator[KMer]:
        if self._written:
            with open(self.tmp, "rt") as th:
                for rec in _simple_fasta(th):
                    yield KMer.from_fasta(rec, self.natype)
        else:
            yield from self._records(do_sort=False)

    def sorted(self, smart: bool = False) -> List[KMer]:
        return list(self._records(do_sort=True))

    def write(self, doSort: bool = False, force: bool = False) -> None:
        """Export as a reference-format batch file: FASTA, one k-mer per record (batch.py:281-296).
        Sorted export (what `kmer batch` asks for) is formatted on the GPU; the unsorted record order
        is only produced for callers that insist on it."""
        if not self._written or force:
            if doSort:
                with open(self.tmp, "wb") as th:
                    self._eng.write_batch(self.device_input, self.k, self.strand_rule, th)
            else:
                with open(self.tmp, "w+") as th:
                    for r in self._records(do_sort=False):
                        th.write(r.as_fasta())
            self._written = True

    def unwrite(self) -> None:
        if self._written and os.path.isfile(self.tmp):
            os.remove(self.tmp)
        self._written = False

    def reset(self) -> None:
        self.unwrite()
        self._n = None


class LoadedKmerBatch(DeviceBatch):
    """Reference-format batch files (`kmer batch` output, kmermaid/batch.py:281-296: ">ref:start-end:strand\nSEQ\n"
    records) re-imported as device keys -- the `-B` reload of `kmer count` / `kmer uniq`
    (kmermaid/batcher.py:616-636, batch.py:298-344).

    Every stored k-mer becomes one record of k bases in a flat base buffer ("SEQ\n" is exactly the
    record + separator layout of the device path), so the extraction kernel at window length k packs
    one key per stored k-mer and its payload (window start) / (k + 1) is the index of the k-mer's
    header.  Reverse complements were materialised when the batches were made, so nothing is
    complemented again."""

    def __init__(self, engine, paths: List[str], natype: NATYPES, tmp_dir: str, alphabet: Optional[str] = None):
        import gzip

        from kman_b200 import fasta

        raw = []
        for path in paths:
            opener = gzip.open if path.endswith(".gz") else open
            with opener(path, "rb") as fh:
                b = fh.read()
            if b and not b.endswith(b"\n"):
                b += b"\n"
            raw.append(b)
        buf = np.frombuffer(b"".join(raw), np.uint8)
        nl = np.flatnonzero(buf == 10)
        if nl.size % 2 or nl.size == 0:
            raise AssertionError("batch files must hold two-line records (>header / sequence)")
        starts = np.concatenate(([0], nl[:-1] + 1))
        h_b, h_e = starts[0::2], nl[0::2]  # header lines (with '>')
        s_b, s_e = starts[1::2], nl[1::2]  # sequence lines
        if not (buf[h_b] == ord(">")).all():
            raise AssertionError("batch files must hold two-line records (>header / sequence)")
        lens = s_e - s_b
        k = int(lens[0])
        if k < 2 or not (lens == k).all():
            raise AssertionError("batch files must hold k-mers of one length")
        n = int(lens.size)
        # flat base buffer: "SEQ\n" per stored k-mer
        idx = (s_b[:, None] + np.arange(k + 1)[None, :]).reshape(-1)
        bases = buf[idx]
        self._hdr_buf = buf
        self._hdr_b, self._hdr_e = h_b + 1, h_e  # without '>'
        flat = fasta.FlatInput(bases, np.array([0, bases.size], np.uint64), ["batch"], ["batch"])
        d = engine.upload(flat, alphabet, natype, with_names=False)
        super().__init__(engine, d, k, False, natype, tmp_dir, size=max(2, n))
        self._n = n
        self.paths = list(paths)

    def uniq_text(self) -> bytes:
        """">HEADER\nSEQ\n" of the k-mers that occur once, ascending by sequence (join.py:243-263), with the
        headers the batch files stored."""
        eng, d, k = self._eng, self.device_input, self.k
        streams = eng.uniq(d, k, False)
        keys = [s.keys_host() for s in streams]
        rec = [(s.vals_host().astype(np.int64) >> 1) // (k + 1) for s in streams]
        txt = [decode_keys(kk, k, s.wide, self.natype) for kk, s in zip(keys, streams)]
        if len(streams) == 2 and streams[1].n and streams[0].n:
            rn, rw = eng.merge_ranks(streams[0].keys, streams[0].n, streams[1].keys, streams[1].n, k, d.rna)
            pos = [np.arange(streams[0].n) + rn.cpu().numpy(), np.arange(streams[1].n) + rw.cpu().numpy()]
            total = streams[0].n + streams[1].n
            order_rec, order_txt = np.empty(total, np.int64), np.empty((total, k), np.uint8)
            for p_, r_, t_ in zip(pos, rec, txt):
                order_rec[p_], order_txt[p_] = r_, t_
        else:
            i = 1 if (len(streams) == 2 and streams[1].n) else 0
            order_rec, order_txt = rec[i], txt[i]
        m = order_rec.shape[0]
        if m == 0:
            return b""
        hb, hl = self._hdr_b[order_rec], (self._hdr_e - self._hdr_b)[order_rec]
        line = hl + k + 3  # '>' header '\n' seq '\n'
        off = np.concatenate(([0], np.cumsum(line)))
        out = np.empty(int(off[-1]), np.uint8)
        out[off[:-1]] = ord(">")
        # ragged copy of the headers: for every output byte of a header, its source index
        tot_h = int(hl.sum())
        within = np.arange(tot_h) - np.repeat(np.cumsum(hl) - hl, hl)
        out[np.repeat(off[:-1] + 1, hl) + within] = self._hdr_buf[np.repeat(hb, hl) + within]
        out[off[:-1] + 1 + hl] = 10
        seq_at = off[:-1] + 2 + hl
        out[(seq_at[:, None] + np.arange(k)[None, :]).reshape(-1)] = order_txt.reshape(-1)
        out[seq_at + k] = 10
        return out.tobytes()
