"""CPU oracle for the kmermaid hot path (extract -> sort -> uniq/count).

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, the smoke check in
__graft_entry__.smoke() and the cpu_baseline / --impl reference legs of bench.py
may import it; nothing under kman_b200/ does.  It restates, on the CPU, what the
reference does on its one correct configuration (SURVEY.md §0: `--scan-mode
KMERS`, `--threads 1`, `kmer uniq` / `kmer count -m SEQ_COUNT`).

Parity status: PINNED for ACGT/acgt input (every golden vector under
tests/golden/ was produced by running the UNMODIFIED reference package with
oracle/gen_golden.py, and tests/test_oracle_golden.py checks this file against
all of them plus the reference's own known-answer tests).  "PARITY UNPINNED" for
the *contents* of the non-ACGT alphabet: that constant lives in the un-vendored
dependency oligo_melting 2.0.1.post3 (git 301b2c84), which is not in
/root/reference.  Both plausible alphabets are implemented as data
(ALPHABETS["IUPAC"] -- upstream's best-known value, the default -- and
ALPHABETS["ACGT"]) and goldens exist for both.

Two tiers, cross-checked against each other in the CPU test-suite:
  * tier A (`*_py`): literal pure-Python restatement, string k-mers, Python
    `sorted`, `heapq.merge`, grouping loop.  Small inputs only.
  * tier B (`*_np`): numpy restatement on packed integer keys.  Used for
    Mbp-scale inputs and as the `cpu_baseline` of bench.py (count_table_np_threads: the
    same stages on all host threads, chunked and merged the way `kmer batch --threads N` is).

Reference citations are relative to /root/reference/.
"""
from __future__ import annotations

import heapq
from typing import Dict, Iterable, Iterator, List, Optional, Sequence, Tuple

import numpy as np

# --------------------------------------------------------------------------------------
# Alphabets (oligo_melting.AB_NA stand-in; kmermaid/seq.py:318 is the only consumer of
# its content, kmermaid/seq.py:279 (mkrc) of the complement row).
# --------------------------------------------------------------------------------------
ALPHABETS: Dict[str, Dict[str, Tuple[str, str]]] = {
    "IUPAC": {
        "DNA": ("ACGTRYKMSWBDHVN", "TGCAYRMKSWVHDBN"),
        "RNA": ("ACGURYKMSWBDHVN", "UGCAYRMKSWVHDBN"),
    },
    "ACGT": {"DNA": ("ACGT", "TGCA"), "RNA": ("ACGU", "UGCA")},
}
DEFAULT_ALPHABET = "IUPAC"

Record = Tuple[str, str]  # (title, sequence) exactly as the reference's parser yields them


# --------------------------------------------------------------------------------------
# FASTA text rules -- kmermaid/parsers.py:53-128 (SmartFastaParser), text-mode newlines
# --------------------------------------------------------------------------------------
def parse_fasta_text(text: str) -> List[Record]:
    """Restates SmartFastaParser.parse (parsers.py:86-128) on an in-memory string.

    * everything before the first line starting with '>' is skipped (parsers.py:53-66);
      no such line -> AssertionError (parsers.py:100-102)
    * title = line[1:].rstrip() (parsers.py:120)
    * sequence = following lines, each rstrip()ed, joined, then " " and "\\r" removed
      (parsers.py:82,124); a line whose first character is '>' starts the next record
    * an empty record terminates here (the reference never returns, SURVEY Appendix A6)
    """
    # the reference reads in text mode with universal newlines
    lines = text.replace("\r\n", "\n").replace("\r", "\n").split("\n")
    if lines and lines[-1] == "":
        lines.pop()  # split() artefact of a trailing newline
    i = 0
    while i < len(lines) and not lines[i].startswith(">"):
        i += 1
    if i == len(lines):
        raise AssertionError("premature end of file or empty file")
    records: List[Record] = []
    while i < len(lines):
        title = lines[i][1:].rstrip()
        i += 1
        seq_lines = []
        while i < len(lines) and not lines[i].startswith(">"):
            seq_lines.append(lines[i].rstrip())
            i += 1
        records.append((title, "".join(seq_lines).replace(" ", "").replace("\r", "")))
    return records


def read_fasta(path: str) -> List[Record]:
    import gzip

    if path.endswith(".gz"):  # batcher.py:480
        with gzip.open(path, "rt", encoding="latin-1", newline="") as fh:
            return parse_fasta_text(fh.read())
    with open(path, "r", encoding="latin-1", newline="") as fh:
        return parse_fasta_text(fh.read())


def record_name(title: str) -> str:
    """batcher.py:551 -- name is the title up to the first SPACE (a TAB stays)."""
    return title.split(" ")[0]


# --------------------------------------------------------------------------------------
# Known-answer helpers restating kmermaid/seq.py
# --------------------------------------------------------------------------------------
def batcher_py(seq: str, k: int, batch_size: int) -> Iterator[Tuple[str, int]]:
    """Sequence.batcher, seq.py:361-383: chunks advancing by batch_size-k+1 (k-1 overlap)."""
    start = 0
    while start < len(seq) - k + 1:
        end = min(len(seq), start + batch_size)
        yield (seq[start:end], start)
        start += batch_size - k + 1


def mkrc_py(s: str, ab: Tuple[str, str]) -> str:
    """om.Sequence.mkrc as used at seq.py:279: reverse, then complement through ab[0]->ab[1]."""
    table = dict(zip(ab[0], ab[1]))
    return "".join(table[c] for c in reversed(s.upper()))


def kmers_py(
    seq: str,
    k: int,
    prefix: str = "ref",
    offset: int = 0,
    rc: bool = False,
    alphabet: str = DEFAULT_ALPHABET,
    natype: str = "DNA",
) -> Iterator[Tuple[str, int, int, str, str]]:
    """Sequence.yield_kmers, seq.py:284-328 (+ rc seq.py:245-282).

    Yields (ref, start, end, strand, kmer_seq) in the reference's order: position
    ascending; with rc the '+' k-mer is followed by its reverse complement carrying the
    SAME coordinates and strand '-'.
    """
    ab = ALPHABETS[alphabet][natype]
    allowed = set(ab[0])
    seq = seq.upper()  # seq.py:313
    for i in range(len(seq) - k + 1):  # seq.py:317
        window = seq[i : i + k]
        if not set(window) <= allowed:  # seq.py:318 check_ab
            continue  # seq.py:319-327 (one WARNING per skipped window, not reproduced)
        yield (prefix, i + offset, i + offset + k, "+", window)  # seq.py:236-243
        if rc:
            yield (prefix, i + offset, i + offset + k, "-", mkrc_py(window, ab))  # seq.py:275-282


def header_py(ref: str, start: int, end: int, strand: str) -> str:
    """SequenceCoords.__repr__, seq.py:103-104."""
    return "%s:%d-%d:%s" % (ref, start, end, strand)


# --------------------------------------------------------------------------------------
# Tier A: literal pipeline
# --------------------------------------------------------------------------------------
def batches_py(
    records: Sequence[Record],
    k: int,
    rc: bool = False,
    batch_size: int = 1_000_000,
    alphabet: str = DEFAULT_ALPHABET,
    natype: str = "DNA",
) -> List[List[Tuple[str, str]]]:
    """FastaBatcher.do in KMERS mode at 1 thread (batcher.py:371-392,535-569,118-153).

    Returns the list of batches; each batch is a list of (header, seq) sorted by seq with
    Python's stable sort (batch.py:156-168), batches filled in input order across records.
    """
    if k <= 1:
        raise AssertionError(f"k must be >= 1, got {k} instead.")  # batcher.py:477-478
    flat: List[Tuple[str, str]] = []
    for title, seq in records:
        name = record_name(title)
        for ref, s, e, strand, kseq in kmers_py(seq, k, name, 0, rc, alphabet, natype):
            flat.append((header_py(ref, s, e, strand), kseq))
    batches = [flat[i : i + batch_size] for i in range(0, len(flat), batch_size)]
    return [sorted(b, key=lambda r: r[1]) for b in batches]


def crawl_groups_py(batches: Sequence[Sequence[Tuple[str, str]]]) -> Iterator[Tuple[List[str], str]]:
    """Crawler.do_records + do_batch, join.py:63-130: n-way merge then run-length grouping."""
    merged = heapq.merge(*batches, key=lambda r: r[1])  # join.py:93
    current_seq: Optional[str] = None
    headers: List[str] = []
    for header, seq in merged:
        if current_seq is None:
            current_seq, headers = seq, [header]
        elif seq == current_seq:
            headers.append(header)
        else:
            yield headers, current_seq
            current_seq, headers = seq, [header]
    if current_seq is not None:
        yield headers, current_seq


def count_text_py(records, k, rc=False, batch_size=1_000_000, alphabet=DEFAULT_ALPHABET, natype="DNA") -> bytes:
    """`kmer count` (SEQ_COUNT) output bytes: join.py:265-285."""
    out = []
    for headers, seq in crawl_groups_py(batches_py(records, k, rc, batch_size, alphabet, natype)):
        out.append("%s\t%d\n" % (seq, len(headers)))
    return "".join(out).encode("latin-1")


def uniq_text_py(records, k, rc=False, batch_size=1_000_000, alphabet=DEFAULT_ALPHABET, natype="DNA") -> bytes:
    """`kmer uniq` output bytes: join.py:243-263 (only groups with exactly one header)."""
    out = []
    for headers, seq in crawl_groups_py(batches_py(records, k, rc, batch_size, alphabet, natype)):
        if len(headers) == 1:
            out.append(">%s\n%s\n" % (headers[0], seq))
    return "".join(out).encode("latin-1")


def batch_text_py(records, k, rc=False, batch_size=1_000_000, alphabet=DEFAULT_ALPHABET, natype="DNA") -> List[bytes]:
    """`kmer batch` file contents (one bytes object per batch): seq.py:489-495, batch.py:281-296."""
    return [
        "".join(">%s\n%s\n" % r for r in b).encode("latin-1")
        for b in batches_py(records, k, rc, batch_size, alphabet, natype)
    ]


# --------------------------------------------------------------------------------------
# Tier B: numpy on packed keys
# --------------------------------------------------------------------------------------
# Order-preserving codes.  For equal-length upper-case strings, Python's str order is code
# point order, so any code that is monotone in ASCII preserves batch.py:156-168's order.
_SYMBOLS16 = "ABCDGHKMNRSTUVWY"  # the 16 IUPAC letters (+U) in ASCII order -> 4-bit rank


def _lut2(natype: str) -> np.ndarray:
    """ASCII -> 2-bit code for the four plain bases (A<C<G<T/U), 0xFF otherwise; case-folded."""
    lut = np.full(256, 0xFF, np.uint8)
    for i, c in enumerate("ACG" + ("T" if natype == "DNA" else "U")):
        lut[ord(c)] = i
        lut[ord(c.lower())] = i
    return lut


def _lut4(alphabet: str, natype: str) -> np.ndarray:
    """ASCII -> 4-bit ASCII-rank code for every symbol of the alphabet, 0xFF otherwise."""
    lut = np.full(256, 0xFF, np.uint8)
    for c in ALPHABETS[alphabet][natype][0]:
        lut[ord(c)] = _SYMBOLS16.index(c)
        lut[ord(c.lower())] = _SYMBOLS16.index(c)
    return lut


def concat_records(records: Sequence[Record]) -> Tuple[np.ndarray, np.ndarray, List[str]]:
    """Flat base buffer: records joined by one '\\n' separator (never a valid symbol, so no
    window spans two records -- batcher.py:387-388 extracts each record on its own).

    Returns (bases u8[n], rec_starts i64[n_rec+1] (start offset of each record in `bases`;
    last entry = one past the end + 1), names)."""
    names = [record_name(t) for t, _ in records]
    parts = []
    starts = np.zeros(len(records) + 1, np.int64)
    pos = 0
    for i, (_, s) in enumerate(records):
        starts[i] = pos
        b = s.encode("latin-1")
        parts.append(b)
        parts.append(b"\n")
        pos += len(b) + 1
    starts[len(records)] = pos
    bases = np.frombuffer(b"".join(parts), np.uint8) if parts else np.zeros(0, np.uint8)
    return bases, starts, names


def _window_all(flag: np.ndarray, k: int) -> np.ndarray:
    """window_ok[i] = all(flag[i:i+k]) for i in [0, len-k]; empty if len < k."""
    n = flag.shape[0]
    if n < k:
        return np.zeros(0, bool)
    bad = np.concatenate(([0], np.cumsum(~flag, dtype=np.int64)))
    return (bad[k:] - bad[:-k]) == 0


def _roll_pack(codes: np.ndarray, k: int, bits: int) -> List[np.ndarray]:
    """Pack k consecutive `bits`-wide codes MSB-first into little-endian-ordered limbs.

    Returns limbs [hi, ..., lo] of uint64 arrays of length len(codes)-k+1 such that the
    window value is sum(limb[j] << 64*(L-1-j)).  Plain shift/or, vectorised over windows.
    """
    n = codes.shape[0] - k + 1
    per = 64 // bits  # symbols per limb
    n_limbs = (k + per - 1) // per
    limbs = []
    # the LOW limb holds the last `per` symbols, and so on upwards
    for li in range(n_limbs):
        hi_sym = k - li * per  # exclusive symbol index end for this limb
        lo_sym = max(0, hi_sym - per)
        acc = np.zeros(n, np.uint64)
        for j in range(lo_sym, hi_sym):
            acc = (acc << np.uint64(bits)) | codes[j : j + n].astype(np.uint64)
        limbs.append(acc)
    return limbs[::-1]


def extract_np(
    records: Sequence[Record],
    k: int,
    rc: bool = False,
    alphabet: str = DEFAULT_ALPHABET,
    natype: str = "DNA",
):
    """Restates seq.py:284-328 for all records at once on the flat buffer.

    Returns a dict with two streams, each in the reference's emission order (record,
    position, '+' before '-'):
      'narrow': windows made only of the four plain bases -> 2-bit packed keys
                keys  : list of uint64 limb arrays [hi, lo] (hi absent when k<=32)
                pos   : int64 global window start in the flat buffer
                strand: uint8 0 '+', 1 '-'
      'wide'  : windows that pass the alphabet test but contain >=1 other symbol ->
                4-bit ASCII-rank keys (same fields)
    plus 'bases', 'rec_starts', 'names', 'n_windows' (all windows, valid or not).
    """
    if k <= 1:
        raise AssertionError(f"k must be >= 1, got {k} instead.")
    bases, rec_starts, names = concat_records(records)
    lut2, lut4 = _lut2(natype), _lut4(alphabet, natype)
    c2, c4 = lut2[bases], lut4[bases]
    ok2 = _window_all(c2 != 0xFF, k)
    ok4 = _window_all(c4 != 0xFF, k)
    n_windows = int(sum(max(0, len(s) - k + 1) for _, s in records))
    out = {"bases": bases, "rec_starts": rec_starts, "names": names, "n_windows": n_windows, "k": k}
    comp_row = ALPHABETS[alphabet][natype]
    comp4 = np.zeros(16, np.uint8)
    for a, b in zip(*comp_row):
        comp4[_SYMBOLS16.index(a)] = _SYMBOLS16.index(b)

    for name, ok, codes, bits in (("narrow", ok2, c2, 2), ("wide", ok4 & ~ok2 if ok2.size else ok4, c4, 4)):
        pos = np.flatnonzero(ok).astype(np.int64)
        if pos.size == 0:
            n_l = (k + (64 // bits) - 1) // (64 // bits)
            out[name] = {"keys": [np.zeros(0, np.uint64)] * n_l, "pos": pos, "strand": np.zeros(0, np.uint8), "bits": bits}
            continue
        safe = np.where(codes == 0xFF, 0, codes)
        fwd = [l[pos] for l in _roll_pack(safe, k, bits)]
        if not rc:
            out[name] = {"keys": fwd, "pos": pos, "strand": np.zeros(pos.size, np.uint8), "bits": bits}
            continue
        # reverse complement: complement each symbol then reverse the window (seq.py:279)
        if bits == 2:
            comp = (np.uint8(3) - safe).astype(np.uint8)  # A<->T, C<->G under A<C<G<T
        else:
            comp = comp4[safe & 0x0F]
        # R = comp reversed; the rc of window [p, p+k) is R[n-k-p : n-p] read forwards
        rev = [l[(bases.shape[0] - k) - pos] for l in _roll_pack(comp[::-1].copy(), k, bits)]
        keys = [np.stack([f, r], axis=1).reshape(-1) for f, r in zip(fwd, rev)]
        out[name] = {
            "keys": keys,
            "pos": np.repeat(pos, 2),
            "strand": np.tile(np.array([0, 1], np.uint8), pos.size),
            "bits": bits,
        }
    return out


def _lexsort_limbs(limbs: List[np.ndarray]) -> np.ndarray:
    """Stable argsort by multi-limb key (batch.py:156-168: stable sort by sequence)."""
    if len(limbs) == 1:
        return np.argsort(limbs[0], kind="stable")
    return np.lexsort(tuple(limbs[::-1]))  # last key is primary; lexsort is stable


def _decode(limbs: List[np.ndarray], k: int, bits: int, natype: str) -> np.ndarray:
    """keys -> (n, k) uint8 ASCII matrix."""
    n = limbs[0].shape[0]
    per = 64 // bits
    sym = np.frombuffer((("ACG" + ("T" if natype == "DNA" else "U")) if bits == 2 else _SYMBOLS16).encode(), np.uint8)
    out = np.empty((n, k), np.uint8)
    L = len(limbs)
    for j in range(k):
        from_end = k - 1 - j  # symbol index counted from the least-significant end
        limb = limbs[L - 1 - from_end // per]
        sh = np.uint64(bits * (from_end % per))
        out[:, j] = sym[((limb >> sh) & np.uint64((1 << bits) - 1)).astype(np.intp)]
    return out


def _rle(limbs: List[np.ndarray]):
    """Crawler.do_batch, join.py:95-130, on sorted packed keys: run heads and lengths."""
    n = limbs[0].shape[0]
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    diff = np.zeros(n - 1, bool)
    for l in limbs:
        diff |= l[1:] != l[:-1]
    heads = np.concatenate(([0], np.flatnonzero(diff) + 1)).astype(np.int64)
    lens = np.diff(np.concatenate((heads, [n]))).astype(np.int64)
    return heads, lens


def _merge_order(a_txt: np.ndarray, b_txt: np.ndarray) -> np.ndarray:
    """Merge two ASCII-sorted (n,k) matrices with no common rows; returns for the merged
    sequence an index array: i>=0 -> a_txt[i], i<0 -> b_txt[-i-1]."""
    k = a_txt.shape[1] if a_txt.size else b_txt.shape[1]
    va = np.ascontiguousarray(a_txt).view("S%d" % k).reshape(-1)
    vb = np.ascontiguousarray(b_txt).view("S%d" % k).reshape(-1)
    # NB: 'S' compares as bytes with trailing-NUL stripping; rows never contain NUL
    ra = np.searchsorted(vb, va, side="left") + np.arange(va.size)
    rb = np.searchsorted(va, vb, side="left") + np.arange(vb.size)
    order = np.empty(va.size + vb.size, np.int64)
    order[ra] = np.arange(va.size)
    order[rb] = -np.arange(vb.size) - 1
    return order


def _coords(ex, pos: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    rec = np.searchsorted(ex["rec_starts"], pos, side="right") - 1
    return rec, pos - ex["rec_starts"][rec]


def count_np(records, k, rc=False, alphabet=DEFAULT_ALPHABET, natype="DNA"):
    """`kmer count` in canonical binary form.

    Returns (txt (U,k) uint8 ASCII matrix of distinct k-mers ascending, counts int64[U],
    and the per-stream detail dict used by the GPU parity tests: for each stream the
    sorted distinct key limbs and their counts)."""
    ex = extract_np(records, k, rc, alphabet, natype)
    detail = {}
    mats, cnts = [], []
    for name in ("narrow", "wide"):
        st = ex[name]
        order = _lexsort_limbs(st["keys"])
        srt = [l[order] for l in st["keys"]]
        heads, lens = _rle(srt)
        ukeys = [l[heads] for l in srt]
        detail[name] = {"keys": ukeys, "counts": lens}
        mats.append(_decode(ukeys, k, st["bits"], natype))
        cnts.append(lens)
    order = _merge_order(mats[0], mats[1])
    txt = np.where((order >= 0)[:, None], mats[0][np.maximum(order, 0)] if mats[0].size else 0,
                   mats[1][np.maximum(-order - 1, 0)] if mats[1].size else 0).astype(np.uint8) \
        if order.size else np.zeros((0, k), np.uint8)
    counts = np.where(order >= 0, cnts[0][np.maximum(order, 0)] if cnts[0].size else 0,
                      cnts[1][np.maximum(-order - 1, 0)] if cnts[1].size else 0).astype(np.int64) \
        if order.size else np.zeros(0, np.int64)
    detail["n_windows"] = ex["n_windows"]
    return txt, counts, detail


def count_table_np(records, k, rc=False, alphabet=DEFAULT_ALPHABET, natype="DNA"):
    """The binary (k-mer, count) table of the NARROW stream only -- distinct packed keys ascending
    (limb list) and their multiplicities -- without decoding to text: the stages bench.py's GPU arm
    times (seq.py:284-328 -> batch.py:156-168 -> join.py:95-130), used by its cpu_baseline leg."""
    st = extract_np(records, k, rc, alphabet, natype)["narrow"]
    order = _lexsort_limbs(st["keys"])
    srt = [l[order] for l in st["keys"]]
    heads, lens = _rle(srt)
    return [l[heads] for l in srt], lens


def count_table_np_threads(records, k, rc=False, alphabet=DEFAULT_ALPHABET, natype="DNA", threads: int = 0,
                           batch_size: Optional[int] = None):
    """count_table_np on `threads` host threads -- the shape of the reference's own parallel run
    (`kmer batch --threads N`: batcher.py:454-487 hands Sequence.batcher's chunks, seq.py:361-383, k-1
    overlap, to joblib workers that each extract and sort one batch, batch.py:156-168; the join then
    merges the sorted batches, join.py:63-130).  Here every worker extracts and sorts the keys of its
    chunks (numpy releases the GIL inside its kernels), and the merge is split by KEY RANGE so that it
    runs in parallel too: worker r takes the r-th key range of every sorted batch (two binary searches
    per batch), merges them with a stable sort (timsort on pre-sorted runs = an n-way merge) and
    run-length groups its range; the ranges concatenate in key order.  Same table as count_table_np."""
    import os
    from concurrent.futures import ThreadPoolExecutor

    T = threads if threads > 0 else len(os.sched_getaffinity(0))
    total = sum(len(s) for _, s in records)
    bs = batch_size if batch_size else max(k, -(-total // (4 * T)) + k - 1)  # ~4 batches per worker
    pieces: List[Record] = []
    for title, seq in records:
        for chunk, _start in batcher_py(seq, k, bs):
            pieces.append((title, chunk))
    n_limbs = 1 if k <= 32 else 2

    def sort_batch(piece: Record):
        st = extract_np([piece], k, rc, alphabet, natype)["narrow"]
        order = _lexsort_limbs(st["keys"])
        return [l[order] for l in st["keys"]]

    with ThreadPoolExecutor(T) as pool:
        batches = list(pool.map(sort_batch, pieces))
        # key ranges by the top limb: T equal slices of the key space actually in use
        top_bits = 2 * k - 64 * (n_limbs - 1)
        edges = [(r << top_bits) // T for r in range(1, T)]

        def cuts(b):
            return np.concatenate(([0], np.searchsorted(b[0], np.array(edges, np.uint64), side="left"), [b[0].shape[0]]))

        cut = [cuts(b) for b in batches]

        def merge_range(r: int):
            limbs = [np.concatenate([b[j][c[r]:c[r + 1]] for b, c in zip(batches, cut)]) if batches else np.zeros(0, np.uint64)
                     for j in range(n_limbs)]
            order = _lexsort_limbs(limbs)
            srt = [l[order] for l in limbs]
            heads, lens = _rle(srt)
            return [l[heads] for l in srt], lens

        parts = list(pool.map(merge_range, range(T)))
    keys = [np.concatenate([p[0][j] for p in parts]) for j in range(n_limbs)]
    return keys, np.concatenate([p[1] for p in parts])


def uniq_np(records, k, rc=False, alphabet=DEFAULT_ALPHABET, natype="DNA"):
    """`kmer uniq` in canonical binary form: singletons ascending by sequence.

    Returns (txt (S,k) uint8, rec int64[S], start int64[S], strand uint8[S], names, detail)."""
    ex = extract_np(records, k, rc, alphabet, natype)
    mats, poss, strands = [], [], []
    detail = {}
    for name in ("narrow", "wide"):
        st = ex[name]
        order = _lexsort_limbs(st["keys"])
        srt = [l[order] for l in st["keys"]]
        heads, lens = _rle(srt)
        sel = heads[lens == 1]
        skeys = [l[sel] for l in srt]
        detail[name] = {"keys": skeys, "pos": st["pos"][order][sel], "strand": st["strand"][order][sel]}
        mats.append(_decode(skeys, k, st["bits"], natype))
        poss.append(st["pos"][order][sel])
        strands.append(st["strand"][order][sel])
    order = _merge_order(mats[0], mats[1])

    def pick(a, b, fill):
        if order.size == 0:
            return np.zeros((0,) + a.shape[1:], a.dtype)
        ia, ib = np.maximum(order, 0), np.maximum(-order - 1, 0)
        xa = a[ia] if a.shape[0] else np.full((order.size,) + a.shape[1:], fill, a.dtype)
        xb = b[ib] if b.shape[0] else np.full((order.size,) + b.shape[1:], fill, b.dtype)
        m = order >= 0
        return np.where(m.reshape((-1,) + (1,) * (a.ndim - 1)), xa, xb)

    txt = pick(mats[0], mats[1], 0).astype(np.uint8)
    pos = pick(poss[0], poss[1], 0)
    strand = pick(strands[0], strands[1], 0)
    rec, start = _coords(ex, pos) if pos.size else (np.zeros(0, np.int64), np.zeros(0, np.int64))
    detail["n_windows"] = ex["n_windows"]
    return txt, rec, start, strand, ex["names"], detail


# ---- text emission (join.py:262,284; seq.py:103-104) -----------------------------------
def _digits(v: np.ndarray) -> np.ndarray:
    d = np.ones(v.shape, np.int64)
    t = v.copy()
    while True:
        t = t // 10
        m = t > 0
        if not m.any():
            return d
        d += m


def _put_decimal(buf: np.ndarray, at: np.ndarray, v: np.ndarray, nd: np.ndarray) -> None:
    """Write decimal of v[i] into buf[at[i] : at[i]+nd[i]]."""
    t = v.copy()
    for j in range(int(nd.max()) if nd.size else 0):
        m = nd > j
        buf[at[m] + nd[m] - 1 - j] = (t[m] % 10 + 48).astype(np.uint8)
        t = t // 10


def count_text_np(records, k, rc=False, alphabet=DEFAULT_ALPHABET, natype="DNA") -> bytes:
    txt, counts, _ = count_np(records, k, rc, alphabet, natype)
    return count_text_from(txt, counts, k)


def count_text_from(txt: np.ndarray, counts: np.ndarray, k: int) -> bytes:
    """"SEQ\tCOUNT\n" lines of count_np's (txt, counts)."""
    n = counts.shape[0]
    if n == 0:
        return b""
    nd = _digits(counts)
    ll = k + 1 + nd + 1
    off = np.concatenate(([0], np.cumsum(ll)))[:-1]
    buf = np.empty(int(ll.sum()), np.uint8)
    for j in range(k):
        buf[off + j] = txt[:, j]
    buf[off + k] = 9
    _put_decimal(buf, off + k + 1, counts, nd)
    buf[off + ll - 1] = 10
    return buf.tobytes()


def uniq_text_np(records, k, rc=False, alphabet=DEFAULT_ALPHABET, natype="DNA") -> bytes:
    txt, rec, start, strand, names, _ = uniq_np(records, k, rc, alphabet, natype)
    return uniq_text_from(txt, rec, start, strand, names, k)


def uniq_text_from(txt: np.ndarray, rec: np.ndarray, start: np.ndarray, strand: np.ndarray, names, k: int) -> bytes:
    """">NAME:START-END:STRAND\nSEQ\n" lines of uniq_np's (txt, rec, start, strand, names)."""
    n = rec.shape[0]
    if n == 0:
        return b""
    name_b = [nm.encode("latin-1") for nm in names]
    name_len = np.array([len(b) for b in name_b], np.int64)
    name_off = np.concatenate(([0], np.cumsum(name_len)))
    name_buf = np.frombuffer(b"".join(name_b) + b"\0", np.uint8)
    end = start + k
    ds, de = _digits(start), _digits(end)
    nl = name_len[rec]
    ll = 1 + nl + 1 + ds + 1 + de + 1 + 1 + 1 + k + 1  # > name : s - e : strand \n seq \n
    off = np.concatenate(([0], np.cumsum(ll)))[:-1]
    buf = np.empty(int(ll.sum()), np.uint8)
    buf[off] = ord(">")
    for j in range(int(nl.max())):
        m = nl > j
        buf[off[m] + 1 + j] = name_buf[name_off[rec[m]] + j]
    p = off + 1 + nl
    buf[p] = ord(":")
    _put_decimal(buf, p + 1, start, ds)
    p = p + 1 + ds
    buf[p] = ord("-")
    _put_decimal(buf, p + 1, end, de)
    p = p + 1 + de
    buf[p] = ord(":")
    buf[p + 1] = np.where(strand == 0, ord("+"), ord("-")).astype(np.uint8)
    buf[p + 2] = 10
    for j in range(k):
        buf[p + 3 + j] = txt[:, j]
    buf[p + 3 + k] = 10
    return buf.tobytes()


# ---- abundance vectors: `kmer count -m VEC_COUNT / VEC_COUNT_MASKED` ---------------------------------
# kmermaid/join.py:287-335 (what a group contributes) + abundance.py:92-172 (the per record-and-strand
# vectors and their files).  The reference crashes in these modes as shipped: AbundanceVector.add_count
# calls super().add_count, and the abstract base raises NotImplementedError (abundance.py:123 -> :60,
# SURVEY.md Appendix A4).  Everything else in the two files works; oracle/gen_golden_vec.py runs the
# reference with that one abstract method neutralised at run time and the goldens pin both tiers below.
def vec_count_py(records, k, rc=False, masked=False, alphabet=DEFAULT_ALPHABET, natype="DNA") -> Dict[str, bytes]:
    """Literal tier.  Returns {file name "REF___STRAND.gz": decompressed file content}."""
    data: Dict[str, Dict[str, List[int]]] = {}

    def add_count(ref, strand, pos, count):  # abundance.py:104-146
        vec = data.setdefault(ref, {}).setdefault(strand, [])
        if len(vec) < pos + 1:
            vec.extend([0] * (pos + 1 - len(vec)))
        if vec[pos] != 0:
            raise AssertionError("can't update non-zero count w/o replace")
        vec[pos] = count

    for headers, seq in crawl_groups_py(batches_py(records, k, rc, 1_000_000, alphabet, natype)):
        coords = []
        for h in headers:  # "ref:start-end:strand", greedy ref (seq.py:44-48)
            left, strand = h.rsplit(":", 1)
            ref, span = left.rsplit(":", 1)
            coords.append((ref, strand, int(span.split("-")[0])))
        if not masked:  # join.py:303-308
            for ref, strand, start in coords:
                add_count(ref, strand, start, len(headers))
        elif len(coords) != 1 and len({c[0] for c in coords}) != 1:  # join.py:326-335
            for ref, strand, start in coords:
                add_count(ref, strand, start, sum(1 for c in coords if c[0] != ref))
    out = {}
    for ref, per in data.items():  # abundance.py:162-172
        for strand, vec in per.items():
            out["%s___%s.gz" % (ref, strand)] = b"# k=%d\n" % k + b"".join(b"%d\n" % c for c in vec)
    return out


def vec_count_np(records, k, rc=False, masked=False, alphabet=DEFAULT_ALPHABET, natype="DNA") -> Dict[str, bytes]:
    """numpy tier of vec_count_py: run lengths scattered back through the window positions."""
    ex = extract_np(records, k, rc, alphabet, natype)
    starts = ex["rec_starts"]
    n_flat = int(ex["bases"].shape[0])
    vec = np.zeros((2, n_flat + 1), np.int64)
    names = ex["names"]
    if len(set(names)) != len(names):
        raise AssertionError("can't update non-zero count w/o replace")  # two records write the same vector
    for name in ("narrow", "wide"):
        st = ex[name]
        if st["pos"].size == 0:
            continue
        order = _lexsort_limbs(st["keys"])
        srt = [l[order] for l in st["keys"]]
        pos, strand = st["pos"][order], st["strand"][order].astype(np.int64)
        heads, lens = _rle(srt)
        group = np.repeat(np.arange(heads.size), lens)
        cnt = lens[group]
        if masked:
            rec = np.searchsorted(starts, pos, side="right") - 1
            # members of my group in my own record: pairs (group, record) are contiguous after the stable sort
            gr = group.astype(np.int64) * (len(names) + 1) + rec
            _, inv, same = np.unique(gr, return_inverse=True, return_counts=True)
            cnt = cnt - same[inv]
            keep = cnt > 0
            pos, strand, cnt = pos[keep], strand[keep], cnt[keep]
        vec[strand, pos] = cnt
    out = {}
    for r, nm in enumerate(names):
        b, e = int(starts[r]), int(starts[r + 1]) - 1
        for s_i, label in ((0, "+"), (1, "-")):
            v = vec[s_i, b:e]
            nz = np.flatnonzero(v)
            if nz.size:
                v = v[: int(nz[-1]) + 1]
                out["%s___%s.gz" % (nm, label)] = b"# k=%d\n" % k + b"".join(b"%d\n" % c for c in v.tolist())
    return out


# ---- deterministic synthetic inputs (SURVEY.md §8d / Appendix B) -------------------------
def synth_bases(n: int, seed: int) -> bytes:
    rng = np.random.default_rng(seed)
    return np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)].tobytes()


def synth_fasta_bytes(records: Iterable[Tuple[str, bytes]], width: int = 60) -> bytes:
    out = []
    for title, seq in records:
        out.append(b">" + title.encode() + b"\n")
        arr = np.frombuffer(seq, np.uint8)
        full = (len(arr) // width) * width
        if full:
            m = np.empty((full // width, width + 1), np.uint8)
            m[:, :width] = arr[:full].reshape(-1, width)
            m[:, width] = 10
            out.append(m.tobytes())
        if len(arr) > full:
            out.append(arr[full:].tobytes() + b"\n")
    return b"".join(out)
