"""Positions that do not fit 32 bits.  A genome-size input (and every rank of a multi-GPU run whose shard
starts past 2^31 bases, dist.py) carries 8-byte payloads (global position << 1 | strand) whose upper word
is not zero, base offsets past 2^31 and 2^32 and more than 2^32 windows in one call.

  * small inputs placed at a large DeviceInput.pos_offset: uniq with wide windows (u128 sort_uniq and
    kmg_sort256 with 8-byte payloads) and kmg_extract_parts, against the oracle's positions shifted;
  * 4-byte payloads past 2^31 positions are refused (KMG_ERR_RANGE) by every entry point that stores them;
  * one real input of 2^32 + 0.85 M bases: a few Mbp islands of sequence at the start, across base 2^31
    and across base 2^32, separated by N filler (no window in either stream with alphabet ACGT), and a
    second record that repeats part of the last island.  Its reference is the oracle on the same records
    with each filler cut to 100 N: the windows are the same up to a known shift per island."""
import io

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402
from gpu_util import first_diff, limbs_to_rows, widen  # noqa: E402


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


def _flat(recs):
    from kman_b200 import fasta

    return fasta.from_records(recs)


def _payloads(st, shift) -> np.ndarray:
    """(position + shift) << 1 | strand of an oracle stream; `shift` a scalar or per-window array."""
    return ((st["pos"].astype(np.uint64) + np.asarray(shift, np.uint64)) << np.uint64(1)) | st["strand"].astype(np.uint64)


def _singletons(rows: np.ndarray, vals: np.ndarray):
    """Keys that occur once, ascending, with their payload (rows: (n,) or (n, L) limbs, least significant first)."""
    order = np.argsort(rows, kind="stable") if rows.ndim == 1 else np.lexsort(rows.T)
    sk, sv = rows[order], vals[order]
    ne = (sk[1:] != sk[:-1]) if rows.ndim == 1 else (sk[1:] != sk[:-1]).any(axis=1)
    one = np.ones(len(sk), bool)
    one[1:] &= ne
    one[:-1] &= ne
    return sk[one], sv[one]


def _iupac_records(seed: int, n: int):
    rng = np.random.default_rng(seed)
    b = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    b[n // 2:n // 2 + n // 8] = b[:n // 8]  # repeats: keys that are not singletons
    at = rng.integers(0, n, n // 200)
    b[at] = np.frombuffer(b"RYKMSWBDHVN", np.uint8)[rng.integers(0, 11, at.size)]
    for s in rng.integers(0, n - 100, 10):
        b[s:s + rng.integers(1, 100)] = ord("N")
    return [("chrP first", b[:n // 3].tobytes().decode()), ("chrQ", b[n // 3:].tobytes().decode())]


OFFSETS = [(1 << 31) - 60_000, 2**32 + 3, 2**47 + 5]  # payloads straddle 2^32; past it; far past it


@pytest.mark.parametrize("k", [25, 45])
@pytest.mark.parametrize("rc", [False, True])
def test_uniq_with_wide_windows_at_large_offsets(eng, k, rc):
    """Engine.uniq: the fused narrow path and the wide stream's sort_uniq (16-byte keys at k = 25,
    kmg_sort256 + select_singletons at k = 45), all with 8-byte payloads past 2^32."""
    recs = _iupac_records(k + rc, 200_000)
    *_, det = ko.uniq_np(recs, k, rc, "IUPAC")
    d = eng.upload(_flat(recs), alphabet="IUPAC")
    for off in OFFSETS:
        d.pos_offset = off
        assert d.payload_bytes == 8
        nar, wid = eng.uniq(d, k, rc)
        assert wid.val_bytes == 8 and det["wide"]["pos"].size > 100
        assert first_diff(nar.keys_host(), limbs_to_rows(det["narrow"]["keys"])) == "equal", off
        assert first_diff(nar.vals_host(), _payloads(det["narrow"], off)) == "equal", off
        assert first_diff(wid.keys_host(), limbs_to_rows(widen(det["wide"]["keys"]))) == "equal", off
        assert first_diff(wid.vals_host(), _payloads(det["wide"], off)) == "equal", off


@pytest.mark.parametrize("k,rc", [(25, True), (45, False)])
def test_extract_parts_at_large_offsets(eng, k, rc):
    """kmg_extract_parts with 8-byte payloads past 2^32: the kept keys of a part range are the filtered
    oracle stream, payloads shifted by pos_offset."""
    from kman_b200.engine import wide_part_table

    recs = _iupac_records(50 + k, 150_000)
    ex = ko.extract_np(recs, k, rc, "IUPAC")
    d = eng.upload(_flat(recs), alphabet="IUPAC")
    n_parts = 16
    narrow_c, wide_c = eng.part_counts(d, k, rc, n_parts)
    for off in OFFSETS:
        d.pos_offset = off
        for wide, want_c in ((False, narrow_c), (True, wide_c)):
            st = ex["wide" if wide else "narrow"]
            rows = limbs_to_rows(widen(st["keys"]) if wide else st["keys"])
            r2 = rows[:, None] if rows.ndim == 1 else rows
            if wide:  # top 16 bits (first 4 symbols) -> part
                sh = 4 * k - 16
                top = (r2[:, sh // 64] >> np.uint64(sh % 64)) & np.uint64(0xFFFF)
                part = wide_part_table(d.rna, n_parts)[top.astype(np.int64)].astype(np.int64)
            else:
                sh = 2 * k - 4
                w, o = divmod(sh, 64)
                top = r2[:, w] >> np.uint64(o)
                if o > 60:
                    top = top | (r2[:, w + 1] << np.uint64(64 - o))
                part = (top & np.uint64(15)).astype(np.int64)
            assert np.array_equal(np.bincount(part, minlength=n_parts), want_c)
            vals = _payloads(st, off)
            for lo, hi in ((0, 1), (3, 9), (15, 16), (0, 16)):
                sel = (part >= lo) & (part < hi)
                a = eng.extract_parts(d, k, rc, wide, 8, n_parts, lo, hi, int(sel.sum()))
                assert first_diff(a.keys_host(), rows[sel]) == "equal", (off, wide, lo, hi)
                assert first_diff(a.vals_host(), vals[sel]) == "equal", (off, wide, lo, hi)


def test_four_byte_payloads_past_2_31_positions_are_refused(eng):
    """val_bytes = 4 cannot hold (position << 1 | strand) once (pos_offset + n_bases) << 1 >= 2^32: every
    entry point that stores payloads refuses it (KMG_ERR_RANGE -> ValueError) instead of truncating."""
    import torch

    from kman_b200 import _lib

    recs = _iupac_records(9, 20_000)
    d = eng.upload(_flat(recs), alphabet="ACGT")
    k, n_parts, kb = 31, 2, 8
    n_win = d.n_bases - k + 1
    bufs = [torch.zeros(2 * n_win * kb, dtype=torch.uint8, device=eng.device) for _ in range(n_parts)]
    vbufs = [torch.zeros(2 * n_win * 4, dtype=torch.uint8, device=eng.device) for _ in range(n_parts)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=eng.device)
    vptrs = torch.tensor([b.data_ptr() for b in vbufs], dtype=torch.int64, device=eng.device)
    cursors = torch.zeros(32 * n_parts, dtype=torch.int64, device=eng.device)
    cptrs = torch.tensor([cursors.data_ptr() + 256 * i for i in range(n_parts)], dtype=torch.int64, device=eng.device)
    status = torch.zeros(2, dtype=torch.int32, device=eng.device)
    lib = eng.lib

    def scatter(fn, off):
        common = (d.bases.data_ptr(), d.n_bases, 0, n_win, k, 0, d.lut.data_ptr(), n_parts, ptrs.data_ptr(), vptrs.data_ptr(),
                  kb, 4, off)
        if fn == "plain":
            return lib.kmg_extract_scatter(*common, cursors.data_ptr(), None, 0, eng._stream())
        if fn == "checked":
            return lib.kmg_extract_scatter_checked(*common, cursors.data_ptr(), 2 * n_win, status.data_ptr(), eng._stream())
        return lib.kmg_extract_scatter_shared(*common, cptrs.data_ptr(), 2 * n_win, status.data_ptr(), eng._stream())

    last_ok = (1 << 31) - d.n_bases - 1  # (pos_offset + n_bases) << 1 = 2^32 - 2: every payload fits
    for fn in ("plain", "checked", "shared"):
        for off in (last_ok + 1, 2**32 + 3, 2**47 + 5):
            assert scatter(fn, off) == _lib.KMG_ERR_RANGE, (fn, off)
            assert "val_bytes=4" in lib.kmg_last_error().decode()
        cursors.zero_()
        assert scatter(fn, last_ok) == _lib.KMG_OK, fn
        torch.cuda.synchronize()
    for off in (last_ok + 1, 2**32 + 3):
        d.pos_offset = off
        assert d.payload_bytes == 8
        with pytest.raises(ValueError, match="val_bytes=4"):
            eng.extract(d, k, False, val_bytes=4)
        n, _ = eng.count_windows(d, k)
        with pytest.raises(ValueError, match="val_bytes=4"):
            eng.extract_parts(d, k, False, False, 4, 16, 0, 16, n)
        with pytest.raises(ValueError, match="val_bytes=4"):
            eng.uniq_narrow(d, k, False, val_bytes=4)
    d.pos_offset = last_ok
    assert d.payload_bytes == 4
    ex = ko.extract_np(recs, k, False, "ACGT")
    a = eng.extract(d, k, False, val_bytes=4)
    assert first_diff(a.vals_host().astype(np.uint64), _payloads(ex["narrow"], last_ok)) == "equal"


# ---- one input past 2^32 bases -------------------------------------------------------------------------
FILL = 100  # N filler of the reference records
LA, LB, LC, LT = 1_000_000, 1_300_000, 1_300_000, 200_000  # islands A, B, C and the second record (chrTail)
B0 = (1 << 31) - LB // 2  # island B straddles base 2^31
C0 = (1 << 32) - LC // 2  # island C straddles base 2^32
# k=31 / 45 plus rc: 4.3 G windows, < 4 M valid; a budget of the bases plus a few GB forces several passes


def _island(rng, n: int, copy_from=None) -> np.ndarray:
    b = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    b[n // 2:n // 2 + n // 10] = b[n // 10:n // 5]  # repeats inside the island
    if copy_from is not None:  # and a stretch of another island
        b[n // 5:n // 5 + 50_000] = copy_from[-80_000:-30_000]
    return b


class Big:
    """The 2^32 + 0.85 M-base input, its short twin (fillers of FILL N) and the shift of every island."""

    def __init__(self):
        from kman_b200 import fasta

        rng = np.random.default_rng(4242)
        a = _island(rng, LA)
        b = _island(rng, LB, a)
        c = _island(rng, LC, b)
        tail = c[300_000:300_000 + LT].copy()
        tail[:1000] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 1000)]
        self.islands = {"A": (a, 0), "B": (b, B0), "C": (c, C0)}  # (bases, start in the big record)
        len_big = C0 + LC
        n = len_big + 1 + LT + 1
        bases = np.full(n, ord("N"), np.uint8)
        bases[:LA], bases[B0:B0 + LB], bases[C0:C0 + LC] = a, b, c
        bases[len_big] = fasta.SEP
        bases[len_big + 1:len_big + 1 + LT] = tail
        bases[-1] = fasta.SEP
        self.flat = fasta.FlatInput(bases, np.array([0, len_big + 1, n], np.uint64), ["chrBig", "chrTail"],
                                    ["chrBig island genome", "chrTail"])
        fill = "N" * FILL
        self.short = [("chrBig island genome", a.tobytes().decode() + fill + b.tobytes().decode() + fill + c.tobytes().decode()),
                      ("chrTail", tail.tobytes().decode())]
        # short record start of B / C -> shift to the big record; chrTail's flat start moves by the C shift
        self.sb, self.sc = LA + FILL, LA + FILL + LB + FILL
        self.shift_b, self.shift_c = B0 - self.sb, C0 - self.sc

    def rel_shift(self, start: np.ndarray, rec: np.ndarray) -> np.ndarray:
        """Shift of a record-relative start in the short records to the big ones."""
        s = np.zeros(start.shape, np.int64)
        big = rec == 0
        s[big & (start >= self.sb)] = self.shift_b
        s[big & (start >= self.sc)] = self.shift_c
        return s

    def flat_shift(self, pos: np.ndarray) -> np.ndarray:
        """Shift of a flat position of the short input to the big one."""
        s = np.zeros(pos.shape, np.int64)
        s[pos >= self.sb] = self.shift_b
        s[pos >= self.sc] = self.shift_c  # (chrTail, after chrBig, moves with island C)
        return s


@pytest.fixture(scope="module")
def big(eng):
    import torch

    g = Big()
    d = eng.upload(g.flat, alphabet="ACGT")
    assert d.n_bases > 2**32 and d.payload_bytes == 8
    g.d = d
    yield g
    del g.d, d
    torch.cuda.empty_cache()


def _budget(eng, d, k, rc, mode, passes, chunk_rows=None, text=True):
    """A budget_bytes under which plan_passes(mode) needs about `passes` passes (never below the largest part)."""
    from kman_b200.engine import pass_bytes

    narrow, wide = eng.part_counts(d, k, rc, 256)
    text_bytes = eng._text_plan(d, k, mode, chunk_rows)[1] if text else 0
    n_win = d.n_bases - k + 1
    cost = lambda a, b: pass_bytes(k, mode, a, b, d.payload_bytes, text_bytes, n_win)  # noqa: E731
    target = cost(-(-int(narrow.sum()) // passes), -(-int(wide.sum()) // passes))
    extra = 8 * (d.n_bases + 1) if mode == "vec" else 0  # the resident vector pair
    return max(target, max(cost(int(a), int(b)) for a, b in zip(narrow, wide))) + eng._resident_bytes(d) + extra


BIG_CASES = [(31, False), (31, True), (45, False), (45, True)]


@pytest.mark.parametrize("k,rc", BIG_CASES)
def test_big_uniq_narrow_over_island_windows(eng, big, k, rc):
    """kmg_extract_sort_uniq over the windows of island B (across base 2^31) and of island C (across 2^32):
    > 2^20 keys each, so the fused front end and the local sort with 8-byte payloads."""
    for name in ("B", "C"):
        bases, start = big.islands[name]
        ex = ko.extract_np([("island", bases.tobytes().decode())], k, rc, "ACGT")
        wk, wv = _singletons(limbs_to_rows(ex["narrow"]["keys"]), _payloads(ex["narrow"], start))
        s, n_other = eng.uniq_narrow(big.d, k, rc, win_begin=start, win_end=start + len(bases) - k + 1)
        assert n_other == 0 and s.val_bytes == 8
        assert len(wk) > (1 << 19)
        assert first_diff(s.keys_host(), wk) == "equal", name
        assert first_diff(s.vals_host(), wv) == "equal", name
        assert int(wv.max() >> np.uint64(33)) == (1 if name == "C" else 0)  # positions past 2^32 in island C


@pytest.mark.parametrize("k,rc", BIG_CASES)
def test_big_write_uniq(eng, big, k, rc):
    """Multi-pass kmg_extract_parts over 4.3 G windows; text with coordinates above 2^32."""
    txt, rec, start, strand, names, _ = ko.uniq_np(big.short, k, rc, "ACGT")
    start = start + big.rel_shift(start, rec)
    assert int(start.max()) > 2**32  # record coordinates past 2^32 in the text
    want = ko.uniq_text_from(txt, rec, start, strand, names, k)
    fh = io.BytesIO()
    plan = eng.write_uniq(big.d, k, rc, fh, budget_bytes=_budget(eng, big.d, k, rc, "uniq", 3, 400_000),
                          chunk_rows=400_000)
    got = fh.getvalue()
    assert plan.n_passes >= 2 and plan.n_parts == 256, plan.parts
    assert len(got) == len(want)
    assert got == want


@pytest.mark.parametrize("k,rc", BIG_CASES)
def test_big_write_count_and_histogram(eng, big, k, rc):
    txt, counts, _ = ko.count_np(big.short, k, rc, "ACGT")
    want = ko.count_text_from(txt, counts, k)
    fh = io.BytesIO()
    plan = eng.write_count(big.d, k, rc, fh, budget_bytes=_budget(eng, big.d, k, rc, "count", 3, 400_000),
                           chunk_rows=400_000)
    assert plan.n_passes >= 2, plan.parts
    assert fh.getvalue() == want
    mult, n_kmers = np.unique(counts, return_counts=True)
    want_h = "".join("%d\t%d\n" % mn for mn in zip(mult.tolist(), n_kmers.tolist())).encode()
    assert mult.size > 2
    fh = io.BytesIO()
    plan = eng.write_histogram(big.d, k, rc, fh, budget_bytes=_budget(eng, big.d, k, rc, "histo", 3, text=False))
    assert plan.n_passes >= 2, plan.parts
    assert fh.getvalue() == want_h


@pytest.mark.parametrize("k,rc", BIG_CASES)
def test_big_vectors(eng, big, k, rc):
    """VEC_COUNT / VEC_COUNT_MASKED (Engine._fill_vectors, key-range passes): the islands' slices of the
    device vectors equal the oracle's vectors, and the vectors sum to the oracle's (so they are zero
    everywhere else).  The 4.3 G-entry vectors stay on the device."""
    import torch

    d = big.d
    tail_big = int(d.flat.rec_starts[1])
    for masked in (False, True):
        want = ko.vec_count_np(big.short, k, rc, masked, "ACGT")
        plan = eng.plan_passes(d, k, rc, "vec", _budget(eng, d, k, rc, "vec", 3, text=False), text=False)
        assert plan.n_passes >= 2, plan.parts
        vec, _ = eng._fill_vectors(d, k, rc, masked, plan)
        n = d.n_bases
        total = 0
        for s_i, label in ((0, "+"), (1, "-")):
            dev = vec[s_i * (n + 1):(s_i + 1) * (n + 1)]
            for rec, base in (("chrBig", 0), ("chrTail", tail_big)):
                body = want.get("%s___%s.gz" % (rec, label))
                if body is None:
                    continue
                ref = np.array(body.split(b"\n", 1)[1].split(), dtype=np.int64)
                total += int(ref.sum())
                spans = [(0, LA, 0), (big.sb, LB, B0), (big.sc, LC, C0)] if rec == "chrBig" else [(0, LT, 0)]
                for s0, ln, b0 in spans:  # (short start, length, big start) of each island
                    r = np.zeros(ln, np.int64)
                    seg = ref[s0:s0 + ln]
                    r[:seg.size] = seg
                    got = dev[base + b0:base + b0 + ln].cpu().numpy().astype(np.uint32).astype(np.int64)
                    assert first_diff(got, r) == "equal", (masked, label, rec, b0)
        assert total > 0
        assert int(vec.sum(dtype=torch.int64)) == total, masked  # (counts are < 2^31 here: int32 holds them)
        del vec
        torch.cuda.empty_cache()
