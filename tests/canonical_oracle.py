"""CPU reference of canonical k-mers (`--canonical`, rc = KMG_CANONICAL), built on the two tiers of
oracle/kmer_oracle.py without changing them.

The canonical record of a window is the smaller, in the reference's string order, of the window and its reverse
complement (the alphabet's complement row, as `-r` uses), with the window's coordinates and strand '-' exactly when
the reverse complement is strictly smaller; a palindrome keeps '+'.  Both tiers start from the reference's own `-r`
records (kmer_oracle.kmers_py / extract_np with rc), which carry the window and its reverse complement side by side,
and keep one of each pair:
  * tier A (`*_py`): strings, Python `sorted`, the grouping loop of kmer_oracle.crawl_groups_py.  Small inputs only.
  * tier B (`*_np`): packed keys; the smaller key is the lexicographic minimum of the forward and reverse limbs.
tests/test_cpu_canonical.py checks the tiers against each other and against the `-r` goldens."""
from typing import Iterator, Sequence, Tuple

import numpy as np

import kmer_oracle as ko


# ---- tier A ------------------------------------------------------------------------------------------------
def kmers_py(seq: str, k: int, prefix: str = "ref", offset: int = 0, alphabet: str = ko.DEFAULT_ALPHABET,
             natype: str = "DNA") -> Iterator[Tuple[str, int, int, str, str]]:
    """(ref, start, end, strand, kmer_seq) of every valid window in position order: its canonical k-mer."""
    it = ko.kmers_py(seq, k, prefix, offset, True, alphabet, natype)
    for fwd, rev in zip(it, it):  # '+' record, then its '-' record with the same coordinates
        yield rev if rev[4] < fwd[4] else fwd


def _groups_py(records: Sequence[ko.Record], k: int, alphabet: str, natype: str):
    if k <= 1:
        raise AssertionError(f"k must be >= 1, got {k} instead.")
    flat = []
    for title, seq in records:
        for ref, s, e, strand, kseq in kmers_py(seq, k, ko.record_name(title), 0, alphabet, natype):
            flat.append((ko.header_py(ref, s, e, strand), kseq))
    return ko.crawl_groups_py([sorted(flat, key=lambda r: r[1])])


def count_text_py(records, k, alphabet=ko.DEFAULT_ALPHABET, natype="DNA") -> bytes:
    """`kmer count --canonical` output bytes."""
    return "".join("%s\t%d\n" % (seq, len(h)) for h, seq in _groups_py(records, k, alphabet, natype)).encode("latin-1")


def uniq_text_py(records, k, alphabet=ko.DEFAULT_ALPHABET, natype="DNA") -> bytes:
    """`kmer uniq --canonical` output bytes (canonical k-mers that occur exactly once)."""
    return "".join(">%s\n%s\n" % (h[0], seq) for h, seq in _groups_py(records, k, alphabet, natype)
                   if len(h) == 1).encode("latin-1")


# ---- tier B ------------------------------------------------------------------------------------------------
def extract_np(records, k, alphabet=ko.DEFAULT_ALPHABET, natype="DNA"):
    """kmer_oracle.extract_np's streams with one canonical key per valid window, in position order; strand 1 where
    the reverse complement is strictly smaller."""
    ex = ko.extract_np(records, k, True, alphabet, natype)
    for name in ("narrow", "wide"):
        st = ex[name]
        fwd, rev = [l[0::2] for l in st["keys"]], [l[1::2] for l in st["keys"]]
        less, eq = np.zeros(fwd[0].size, bool), np.ones(fwd[0].size, bool)  # rev < fwd, limbs from the top
        for f, r in zip(fwd, rev):
            less |= eq & (r < f)
            eq &= r == f
        st["keys"] = [np.where(less, r, f) for f, r in zip(fwd, rev)]
        st["pos"] = st["pos"][0::2]
        st["strand"] = less.astype(np.uint8)
    return ex


def _merged(cols, order, fill_shape):
    """Rows of the narrow/wide pair in merged order (kmer_oracle._merge_order's index convention)."""
    a, b = cols
    if order.size == 0:
        return np.zeros((0,) + fill_shape, a.dtype)
    ia, ib = np.maximum(order, 0), np.maximum(-order - 1, 0)
    xa = a[ia] if a.shape[0] else np.zeros((order.size,) + a.shape[1:], a.dtype)
    xb = b[ib] if b.shape[0] else np.zeros((order.size,) + b.shape[1:], b.dtype)
    return np.where((order >= 0).reshape((-1,) + (1,) * (a.ndim - 1)), xa, xb)


def count_np(records, k, alphabet=ko.DEFAULT_ALPHABET, natype="DNA"):
    """(txt (U,k) uint8 canonical k-mers ascending, counts int64[U], per-stream detail) as kmer_oracle.count_np."""
    ex = extract_np(records, k, alphabet, natype)
    detail, mats, cnts = {}, [], []
    for name in ("narrow", "wide"):
        st = ex[name]
        order = ko._lexsort_limbs(st["keys"])
        srt = [l[order] for l in st["keys"]]
        heads, lens = ko._rle(srt)
        ukeys = [l[heads] for l in srt]
        detail[name] = {"keys": ukeys, "counts": lens}
        mats.append(ko._decode(ukeys, k, st["bits"], natype))
        cnts.append(lens)
    order = ko._merge_order(mats[0], mats[1])
    detail["n_windows"] = ex["n_windows"]
    return (_merged(mats, order, (k,)).astype(np.uint8), _merged(cnts, order, ()).astype(np.int64),
            detail)


def uniq_np(records, k, alphabet=ko.DEFAULT_ALPHABET, natype="DNA"):
    """(txt, rec, start, strand, names, detail) of the canonical singletons, as kmer_oracle.uniq_np."""
    ex = extract_np(records, k, alphabet, natype)
    detail, mats, poss, strands = {}, [], [], []
    for name in ("narrow", "wide"):
        st = ex[name]
        order = ko._lexsort_limbs(st["keys"])
        srt = [l[order] for l in st["keys"]]
        heads, lens = ko._rle(srt)
        sel = heads[lens == 1]
        skeys = [l[sel] for l in srt]
        detail[name] = {"keys": skeys, "pos": st["pos"][order][sel], "strand": st["strand"][order][sel]}
        mats.append(ko._decode(skeys, k, st["bits"], natype))
        poss.append(st["pos"][order][sel])
        strands.append(st["strand"][order][sel])
    order = ko._merge_order(mats[0], mats[1])
    txt = _merged(mats, order, (k,)).astype(np.uint8)
    pos = _merged(poss, order, ())
    strand = _merged(strands, order, ())
    rec, start = ko._coords(ex, pos) if pos.size else (np.zeros(0, np.int64), np.zeros(0, np.int64))
    detail["n_windows"] = ex["n_windows"]
    return txt, rec, start, strand, ex["names"], detail


def count_text_np(records, k, alphabet=ko.DEFAULT_ALPHABET, natype="DNA") -> bytes:
    txt, counts, _ = count_np(records, k, alphabet, natype)
    return ko.count_text_from(txt, counts, k)


def uniq_text_np(records, k, alphabet=ko.DEFAULT_ALPHABET, natype="DNA") -> bytes:
    txt, rec, start, strand, names, _ = uniq_np(records, k, alphabet, natype)
    return ko.uniq_text_from(txt, rec, start, strand, names, k)
