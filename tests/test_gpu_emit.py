"""K6 against host formatters: kmg_format_counts / kmg_format_uniq byte for byte against Python's own
`%` formatting of the same rows, the narrow/wide merge ranks (kmg_merge_ranks / kmg_merge_ranks_wide)
against `bisect` on the decoded strings, and RNA inputs end to end (write_count / write_uniq) against
the oracle.  Inputs are synthetic rows built here, so every digit length, key width, record layout and
merge edge is reached on purpose rather than by chance."""
import bisect
import io

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402

SYMBOLS16 = "ABCDGHKMNRSTUVWY"  # 4-bit code -> letter (wide keys); plain bases are 2-bit ACGT / ACGU


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


def _dev(eng, arr: np.ndarray):
    import torch

    return torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1).copy()).to(eng.device)


def _pack(codes: np.ndarray, bits: int, key_bytes: int) -> np.ndarray:
    """(n, k) symbol codes, first symbol most significant -> (n, key_bytes / 8) uint64 limbs, least
    significant limb first (the device layout of 8-, 16- and 32-byte keys)."""
    n, k = codes.shape
    limbs = np.zeros((n, key_bytes // 8), np.uint64)
    for q in range(k):
        sh = bits * (k - 1 - q)
        w, o = divmod(sh, 64)
        limbs[:, w] |= codes[:, q].astype(np.uint64) << np.uint64(o)
    return limbs


def _ascii(codes: np.ndarray, letters: str) -> list:
    lut = np.frombuffer(letters.encode(), np.uint8)
    return [bytes(r) for r in lut[codes]]


# ---- kmg_format_counts -------------------------------------------------------------------------------
KEY_LAYOUTS = [(8, False), (16, False), (32, False), (8, True), (16, True), (32, True)]  # (key bytes, wide)
COUNT_EDGES = np.array([1, 9, 10, 99, 100, 999, 1000, 65535, 65536, 10**9 - 1, 10**9, 2**31, 2**32 - 2, 2**32 - 1],
                       np.uint64)
SIZES = [1, 1023, 1024, 1025, 3 * 1024 + 7, 300_007]  # rows: one tile of 1024 rows, its edges, many tiles


def _counts(rng, n: int) -> np.ndarray:
    """uint32 counts of every digit length 1..10, the edges of each length among them."""
    nd = rng.integers(1, 11, size=n)
    lo = (10 ** (nd - 1)).astype(np.uint64)
    hi = np.minimum(10 ** nd.astype(np.uint64) - 1, 2**32 - 1).astype(np.uint64)
    c = lo + (rng.random(n) * (hi - lo + 1).astype(np.float64)).astype(np.uint64)
    c = np.minimum(c, hi)
    at = rng.integers(0, n, size=min(n, 2 * COUNT_EDGES.size))
    c[at] = COUNT_EDGES[np.arange(at.size) % COUNT_EDGES.size]
    c[0] = COUNT_EDGES[rng.integers(0, COUNT_EDGES.size)]
    return c.astype(np.uint32)


@pytest.mark.parametrize("key_bytes,wide,k", [(kb, w, k) for kb, w in KEY_LAYOUTS for k in (2, 16, 31, 32, 33, 63, 64)
                                              if k * (4 if w else 2) <= 8 * kb])
def test_format_counts_matches_python(eng, k, key_bytes, wide):
    from kman_b200.engine import CountTable

    bits = 4 if wide else 2
    rng = np.random.default_rng(k * 100 + key_bytes + wide)
    for i, n in enumerate(SIZES):
        for rna in (0, 1):
            if n == SIZES[-1] and rna != k % 2:
                continue  # (the big size once per k)
            codes = rng.integers(0, 1 << bits, size=(n, k), dtype=np.uint8)
            counts = _counts(rng, n)
            letters = SYMBOLS16 if wide else ("ACGU" if rna else "ACGT")
            want = b"".join(s + b"\t%d\n" % c for s, c in zip(_ascii(codes, letters), counts.tolist()))
            shift = (n + rna) % 4  # the text starts 0..3 bytes past a 4-byte boundary
            buf = eng._new(n * (k + 12) + 8)
            t = CountTable(_dev(eng, _pack(codes, bits, key_bytes)), _dev(eng, counts), n, key_bytes, k, wide)
            got = eng.format_counts(t, rna, buf[shift:])
            assert got.data_ptr() % 4 == shift
            got = got.cpu().numpy().tobytes()
            assert len(got) == len(want), (n, rna, len(got), len(want))
            if got != want:
                j = next(j for j in range(len(want)) if got[j] != want[j])
                pytest.fail(f"n={n} rna={rna} first difference at byte {j}: {got[j - 40:j + 40]!r} vs {want[j - 40:j + 40]!r}")


# ---- kmg_format_uniq ---------------------------------------------------------------------------------
def _records(rng, n_rec: int, max_len: int, k: int):
    """rec_starts (uint64, n_rec + 1) from 0: record lengths >= k with a separator after each, a few
    empty records (start equal to the next start) in between; names of 1 to 5000 bytes."""
    lens = rng.integers(k, max_len, size=n_rec)
    empty = rng.random(n_rec) < 0.2
    empty[0] = False
    step = np.where(empty, 0, lens + 1).astype(np.uint64)
    starts = np.concatenate(([0], np.cumsum(step))).astype(np.uint64)
    name_len = rng.integers(1, 5001, size=n_rec)
    name_len[:2] = (1, 5000)
    names = [bytes(rng.integers(33, 127, size=int(m), dtype=np.uint8)).replace(b":", b"_") for m in name_len]
    return starts, names, ~empty


def _format_uniq(eng, keys, vals, n, key_bytes, val_bytes, k, wide, rna, starts, names):
    from kman_b200 import _lib

    offs = np.concatenate(([0], np.cumsum([len(m) for m in names]))).astype(np.int64)
    d_starts, d_names, d_offs = _dev(eng, starts), _dev(eng, np.frombuffer(b"".join(names) + b"\0", np.uint8)), _dev(eng, offs)
    text = eng._new(n * (k + 48 + max(len(m) for m in names)))
    ws_bytes = eng.lib.kmg_format_workspace_bytes(n)
    ws = eng._new(ws_bytes)
    _lib.check(eng.lib.kmg_format_uniq(keys.data_ptr(), vals.data_ptr(), n, key_bytes, val_bytes, k, int(wide), rna,
                                       d_starts.data_ptr(), len(names), d_names.data_ptr(), d_offs.data_ptr(),
                                       text.data_ptr(), eng._small[4:].data_ptr(), ws.data_ptr(), ws_bytes, eng._stream()))
    eng._status(ws)
    nbytes = int(eng._small[4:5].cpu().numpy().view(np.uint64)[0])
    return text[:nbytes].cpu().numpy().tobytes()


@pytest.mark.parametrize("k,key_bytes,wide", [(31, 8, False), (45, 16, False), (25, 16, True), (45, 32, True), (2, 8, False)])
@pytest.mark.parametrize("val_bytes", [4, 8])
def test_format_uniq_matches_python(eng, k, key_bytes, wide, val_bytes):
    """Positions at record starts and at the last window of a record, both strands; empty records; with
    8-byte payloads, record starts and positions above 2^32."""
    rng = np.random.default_rng(k + key_bytes + val_bytes)
    n_rec = 60
    starts, names, nonempty = _records(rng, n_rec, 200_000, k)
    # 4-byte payloads (pos << 1 | strand) must fit 32 bits: the records end just below 2^31; 8-byte ones
    # straddle 2^32
    base = (1 << 31) - 50_000 - int(starts[-1]) if val_bytes == 4 else (1 << 32) - int(starts[-1]) // 2
    starts = starts + np.uint64(base)
    real = np.flatnonzero(nonempty)
    pos, strand = [], []
    for r in real:  # first and last window of every record, both strands, and a few inside
        b, e = int(starts[r]), int(starts[r + 1]) - 1
        for p in (b, e - k, *rng.integers(b, e - k + 1, size=6).tolist()):
            pos += [p, p]
            strand += [0, 1]
    pos, strand = np.array(pos, np.uint64), np.array(strand, np.uint64)
    n = pos.size
    vals = (pos << np.uint64(1)) | strand
    assert val_bytes == 8 or int(vals.max()) < 2**32
    if val_bytes == 8:
        assert int(starts[real[-1]]) > 2**32 and int(pos.min()) < 2**32  # both sides of 2^32
    bits = 4 if wide else 2
    for rna in (0, 1):
        codes = rng.integers(0, 1 << bits, size=(n, k), dtype=np.uint8)
        seqs = _ascii(codes, SYMBOLS16 if wide else ("ACGU" if rna else "ACGT"))
        st = starts[:n_rec].astype(np.int64).tolist()
        want = []
        for p, s, seq in zip(pos.tolist(), strand.tolist(), seqs):
            r = bisect.bisect_right(st, p) - 1
            start = p - st[r]
            want.append(b">%s:%d-%d:%s\n%s\n" % (names[r], start, start + k, b"+-"[s:s + 1], seq))
        want = b"".join(want)
        keys = _dev(eng, _pack(codes, bits, key_bytes))
        got = _format_uniq(eng, keys, _dev(eng, vals.astype(np.uint32 if val_bytes == 4 else np.uint64)), n, key_bytes,
                           val_bytes, k, wide, rna, starts, names)
        assert len(got) == len(want), (rna, len(got), len(want))
        assert got == want, rna


# ---- narrow / wide merge ranks -----------------------------------------------------------------------
def _plain(rna: int) -> str:
    return "ACGU" if rna else "ACGT"


def _wide_strings(rng, k: int, rna: int) -> list:
    """Distinct wide strings, sorted: the first non-plain symbol at every position j with every non-plain
    letter there (plain prefix, any suffix), T..TY / U..UY (T' = 4^k - 1) and a B first (T' = 0)."""
    plain = _plain(rna)
    other = [c for c in SYMBOLS16 if c not in plain]
    out = {plain[3] * (k - 1) + "Y", "B" + "".join(rng.choice(list(SYMBOLS16), size=k - 1))}
    for j in range(k):
        for c in other:
            pre = "".join(rng.choice(list(plain), size=j))
            # a U (RNA) / T (DNA) in the prefix: a plain base in one natype, non-plain in the other
            if j and rng.random() < 0.5:
                pre = pre[:-1] + plain[3]
            out.add(pre + c + "".join(rng.choice(list(SYMBOLS16), size=k - 1 - j)))
    return sorted(out)


def _below(w: str, plain: str) -> int:
    """Number of length-k plain strings that sort below the wide string w."""
    k, t = len(w), 0
    for q, ch in enumerate(w):
        if ch in plain:
            t += plain.index(ch) * 4 ** (k - 1 - q)
            continue
        return t + sum(1 for b in plain if b < ch) * 4 ** (k - 1 - q)
    return t


def _narrow_string(v: int, k: int, plain: str) -> str:
    return "".join(plain[(v >> (2 * (k - 1 - q))) & 3] for q in range(k))


def _limbs(values, n_limbs: int) -> np.ndarray:
    m = (1 << 64) - 1
    return np.array([[(v >> (64 * i)) & m for i in range(n_limbs)] for v in values], np.uint64).reshape(-1, n_limbs)


@pytest.mark.parametrize("k", [2, 3, 16, 31, 32, 33, 48, 63, 64])
@pytest.mark.parametrize("rna", [0, 1])
def test_merge_ranks_match_bisect(eng, k, rna):
    import torch

    rng = np.random.default_rng(k * 2 + rna)
    plain = _plain(rna)
    wide = _wide_strings(rng, k, rna)
    top = 4**k - 1
    near = set()
    for w in wide:  # T' - 1, T', T' + 1 of every wide key (T' = the largest plain string below it)
        t = _below(w, plain) - 1
        near.update(x for x in (t - 1, t, t + 1) if 0 <= x <= top)
    near.update(int(x) for x in rng.integers(0, 4**min(k, 31), size=500))
    near.update((int(x) << (2 * k - 62)) for x in rng.integers(0, 1 << 62, size=500) if k > 31)
    narrow = sorted(x for x in near if 0 <= x <= top)
    nstr = [_narrow_string(v, k, plain) for v in narrow]
    assert nstr == sorted(nstr)
    wcodes = np.array([[SYMBOLS16.index(c) for c in w] for w in wide], np.uint8)
    wkb, nlimbs = (16, 1) if k <= 32 else (32, 2)
    for n_n, n_w in ((len(narrow), len(wide)), (0, len(wide)), (len(narrow), 0)):
        nk = _dev(eng, _limbs(narrow[:n_n] or [0], nlimbs))
        wk = _dev(eng, _pack(wcodes[:max(n_w, 1)], 4, wkb))
        rn, rw = eng.merge_ranks(nk, n_n, wk, n_w, k, rna)
        torch.cuda.synchronize()
        want_w = [bisect.bisect_left(nstr[:n_n], w) for w in wide[:n_w]]
        want_n = [bisect.bisect_left(wide[:n_w], s) for s in nstr[:n_n]]
        got_w, got_n = rw.cpu().numpy().tolist(), rn.cpu().numpy().tolist()
        bad_w = [(wide[i], got_w[i], want_w[i]) for i in range(n_w) if got_w[i] != want_w[i]]
        bad_n = [(nstr[j], got_n[j], want_n[j]) for j in range(n_n) if got_n[j] != want_n[j]]
        assert not bad_w, (n_n, n_w, len(bad_w), bad_w[:3])
        assert not bad_n, (n_n, n_w, len(bad_n), bad_n[:3])


# ---- RNA end to end ------------------------------------------------------------------------------------
def _rna_records(seed: int):
    """U-based random sequence with stray T (in neither RNA alphabet), IUPAC symbols, N runs, soft-masked
    stretches and a repeated stretch (counts > 1), over three records."""
    rng = np.random.default_rng(seed)
    n = 120_000
    b = np.frombuffer(b"ACGU", np.uint8)[rng.integers(0, 4, n)].copy()
    b[60_000:75_000] = b[5_000:20_000]
    at = rng.integers(0, n, n // 400)
    b[at] = np.frombuffer(b"RYKMSWBDHVNT", np.uint8)[rng.integers(0, 12, at.size)]
    for s in rng.integers(0, n - 300, 8):
        b[s:s + rng.integers(1, 300)] = ord("N")
    for s in rng.integers(0, n - 2000, 6):
        b[s:s + 2000] |= 0x20
    return [("rnaA first", b[:50_000].tobytes().decode()), ("rnaB", b[50_000:110_000].tobytes().decode()),
            ("rnaC", b[110_000:].tobytes().decode())]


def _forced_budget(eng, d, k, rc, mode, passes, chunk_rows):
    """A device budget under which plan_passes needs about `passes` passes (never below the largest part)."""
    from kman_b200.engine import pass_bytes

    narrow, wide = eng.part_counts(d, k, rc, 256)
    _, text_bytes = eng._text_plan(d, k, mode, chunk_rows)
    n_win = max(0, d.n_bases - k + 1)
    cost = lambda a, b: pass_bytes(k, mode, a, b, d.payload_bytes, text_bytes, n_win)  # noqa: E731
    target = cost(-(-int(narrow.sum()) // passes), -(-int(wide.sum()) // passes))
    return max(target, max(cost(int(a), int(b)) for a, b in zip(narrow, wide))) + eng._resident_bytes(d)


RNA_RECS = _rna_records(2024)


@pytest.mark.parametrize("alphabet", ["ACGT", "IUPAC"])
@pytest.mark.parametrize("k", [12, 31, 45])
@pytest.mark.parametrize("rc", [False, True])
def test_rna_write_count_and_uniq_match_oracle(eng, alphabet, k, rc):
    from kman_b200 import alphabet as ab, fasta

    d = eng.upload(fasta.from_records(RNA_RECS), alphabet=alphabet, natype=ab.NATYPES.RNA)
    assert d.rna == 1
    for mode, writer, ref in (("count", eng.write_count, ko.count_text_np), ("uniq", eng.write_uniq, ko.uniq_text_np)):
        want = ref(RNA_RECS, k, rc, alphabet, natype="RNA")
        assert b"U" in want and (alphabet == "ACGT" or b"T" not in want.replace(b"\t", b""))
        fh = io.BytesIO()
        plan = writer(d, k, rc, fh, chunk_rows=997)
        assert plan.n_passes == 1 and fh.getvalue() == want, (mode, "one pass")
        fh = io.BytesIO()
        plan = writer(d, k, rc, fh, chunk_rows=997, budget_bytes=_forced_budget(eng, d, k, rc, mode, 4, 997))
        assert plan.n_passes >= 2 and fh.getvalue() == want, (mode, plan.n_passes)
        if alphabet == "IUPAC":
            assert int(plan.wide.sum()) > 0  # the wide stream was split by kmg_wide_part_table(rna=1)
