"""GPU parity: text tokenise+combine kernels (csrc/text.cu) vs the oracle restatement.

Bit-exact: counts, line counts, the '' token, key strings."""
import os

import numpy as np
import pytest

from dampr_b200 import device as dev
from dampr_b200 import keycodes
from oracle import gen, refsem

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=[(2, 3), (2, 4), (2, 2), (1, 2)],
                ids=["kernel-v2-3cta", "kernel-v2-4cta", "kernel-v2-2cta", "kernel-v1"])
def text_kernel(request):
    """Every case runs against both tokenise kernels (text2.cu in its three occupancy variants is the
    default, text.cu the fallback)."""
    dev.set_option("text_kernel", request.param[0])
    dev.set_option("text_ctas", request.param[1])
    yield request.param[0]
    dev.set_option("text_kernel", 2)
    dev.set_option("text_ctas", 4)


def run_count(ctx, data, mode, chunk=None, verify=True):
    tb = ctx.textbuf(len(data) + 64)
    arr = np.frombuffer(data, dtype=np.uint8)
    tb.upload_all(arr)
    tab = ctx.table(20)
    n = len(data)
    if chunk is None:
        tab.count(tb, 0, n, mode)
    else:
        lo = 0
        while lo < n:
            hi = min(n, lo + chunk)
            tab.count(tb, lo, hi, mode)
            lo = hi
    st = tab.stats()
    if verify and st["hashed"]:
        tab.verify(tb, 0, n, mode)
        st = tab.stats()
    codes, counts, reps = tab.fetch()
    words = keycodes.decode_table(codes, reps, mode, lambda off, ln: data[off:off + ln])
    got = dict(zip(words, counts.tolist()))
    assert len(got) == len(words), "two table entries decoded to the same word"
    tb.free()
    tab.free()
    return got, st


def check_wc(ctx, data, **kw):
    got, st = run_count(ctx, data, dev.TOK_WS, **kw)
    exp = refsem.wc_counts(data)
    assert st["flags"] & ~dev.TF_CR == 0, st
    assert got == dict(exp)
    assert st["lines"] == len(refsem.text_lines(data))


def check_df(ctx, data, **kw):
    got, st = run_count(ctx, data, dev.TOK_NONWORD_LOWER_SET, **kw)
    exp, n_lines = refsem.docfreq(data)
    assert st["flags"] == 0, st
    exp = dict(exp)
    empty = exp.pop("", 0)
    assert st["empty"] == empty
    assert st["lines"] == n_lines
    assert got == exp


def check_tf(ctx, data, **kw):
    got, st = run_count(ctx, data, dev.TOK_NONWORD_LOWER, **kw)
    exp = dict(refsem.termfreq_nonset(data))
    empty = exp.pop("", 0)
    assert st["flags"] == 0, st
    assert st["empty"] == empty
    assert got == exp


SMALL = [
    b"", b"\n", b"a", b"a\n", b"a b", b"a\n\n", b"\n\n\n", b" a", b"a. b", b"...", b"...\n",
    b"Hello hello HELLO\nhello world\n", b"x_1 X_1 x-1\n", b"one two  three\t\tfour\n\nfive",
    b"a" * 12 + b" " + b"a" * 13 + b" " + b"A" * 13 + b"\n",
    b"abcdefghi abcdefghij abcdefghij\n", b"tail without newline " * 3,
]


@pytest.mark.parametrize("data", SMALL)
def test_small_cases(ctx, data):
    check_wc(ctx, data)
    check_df(ctx, data)
    check_tf(ctx, data)


def test_synthetic_zipf(ctx):
    data = gen.text(1234, 30000, V=5000)
    check_wc(ctx, data)
    check_df(ctx, data)


def test_synthetic_chunked_ownership(ctx):
    """Ownership ranges split at arbitrary 16-byte multiples must count every line exactly once."""
    data = gen.text(99, 8000, V=2000)
    for chunk in (16, 4096 + 16, 6144, 100000):
        check_df(ctx, data, chunk=chunk)
        check_wc(ctx, data, chunk=chunk)


def test_dirty_corpus(ctx):
    data = gen.dirty_text()
    check_wc(ctx, data)
    check_df(ctx, data)
    check_tf(ctx, data)


def test_tile_boundaries(ctx):
    """Tokens and lines straddling the 6 KB tile seams."""
    rng = np.random.default_rng(5)
    words = [b"w%d" % i for i in range(50)] + [b"LongerWord%d" % i for i in range(20)]
    lines = []
    for _ in range(4000):
        k = int(rng.integers(1, 30))
        lines.append(b" ".join(words[int(rng.integers(0, len(words)))] for _ in range(k)))
    data = b"\n".join(lines) + b"\n"
    check_wc(ctx, data)
    check_df(ctx, data)


def test_flags(ctx, text_kernel):
    _, st = run_count(ctx, "café au lait\n".encode("utf-8"), dev.TOK_WS)
    assert st["flags"] & dev.TF_NONASCII
    _, st = run_count(ctx, b"a\r\nb\r\n", dev.TOK_WS)
    assert st["flags"] & dev.TF_CR          # str.split: scan-wide flag (token counts do not depend on it)
    _, st = run_count(ctx, b"a\r\nb\r\n", dev.TOK_NONWORD_LOWER_SET)
    if text_kernel == 1:
        assert st["flags"] & dev.TF_CR and st["fallback"] == 0   # first generation: '\r' flags the whole scan
    else:
        assert st["flags"] == 0 and st["fallback"] == 2   # [^\w]+ modes: the two lines go to the host, nothing else
    long_line = b"x " * 20000 + b"\n"
    _, st = run_count(ctx, b"a\n" * 4000 + long_line + b"b\n" * 4000, dev.TOK_NONWORD_LOWER_SET)
    assert st["flags"] & dev.TF_LONGLINE    # longer than either kernel's window
    # more distinct tokens in one line than the de-duplication history of the v2 kernel holds
    many = b" ".join(b"w%d" % i for i in range(400)) + b"\n"
    if text_kernel == 2:
        _, st = run_count(ctx, b"a b\n" * 10 + many + b"c\n", dev.TOK_NONWORD_LOWER_SET)
        assert st["flags"] & dev.TF_LONGLINE
    # both are fine for the first-generation kernel when they fit its 4 KB window
    dev.set_option("text_kernel", 1)
    try:
        check_df(ctx, b"a b\n" * 10 + many + b"c\n")
    finally:
        dev.set_option("text_kernel", text_kernel)
    # the whitespace tokeniser has no line dependence: long lines are fine there
    check_wc(ctx, b"a\n" * 4000 + long_line + b"b\n" * 4000)


def test_very_long_token(ctx):
    data = b"short " + b"z" * 20000 + b" tail\n" + b"z" * 20000 + b"\n"
    check_wc(ctx, data)


def test_synth_text_matches_numpy_generator(ctx):
    V = 3000
    vocab = gen.make_vocab(V)
    cdf = gen.make_cdf(V)
    n_lines = 5000
    ref = gen.text(77, n_lines, vocab=vocab, cdf=cdf)
    tb = ctx.textbuf(len(ref) + 4096)
    import ctypes as C
    out = C.c_uint64(0)
    vb, vo = vocab
    ctx.check(ctx.lib.dampr_synth_text(ctx.h, tb.h, 77, n_lines, vb.ctypes.data_as(C.c_void_p),
                                       vo.ctypes.data_as(C.c_void_p), V, cdf.ctypes.data_as(C.c_void_p),
                                       C.byref(out)))
    assert out.value == len(ref)
    tb.n = out.value
    got = tb.download(0, out.value).tobytes()
    assert got == ref


def _bad_line_corpus(seed=3, n_lines=6000):
    """ASCII lines with, every so often, a line the device must hand back: non-ASCII bytes (accents, a dotted
    capital I whose lower() grows, a non-breaking space), '\\r\\n', a lone '\\r' inside, a long line with one
    accent at its very end, bad lines next to each other and as first / last line."""
    rng = np.random.default_rng(seed)
    base = gen.text(seed, n_lines, V=3000).rstrip(b"\n").split(b"\n")
    special = ["naïve café".encode(), b"cr inside\rline two", b"crlf line\r", "ÜBER İstanbul straße".encode(),
               "nbsp\u00a0separated words".encode(), b"x " * 700 + "é".encode(), b"\r", "é".encode(), b"a\rb\rc\r"]
    lines = []
    for i, l in enumerate(base):
        if i % 97 == 0:
            lines.append(special[(i // 97) % len(special)])
            if i % (97 * 4) == 0:
                lines.append(special[(i // 97 + 3) % len(special)])   # two bad lines in a row
        lines.append(l)
    lines.append(special[0])                                            # ... and one as the last line
    return lines


def test_per_line_fallback_lists_exactly_the_bad_lines(ctx, text_kernel):
    """[^\\w]+ tokenisers: a line holding a byte the device cannot tokenise like Python (non-ASCII, '\\r' in text
    mode) contributes nothing to the table / line count / '' count and is reported with its offset and length;
    everything else is counted as if those lines were not there. The first-generation kernel keeps no such list: any
    such byte (a '\\r' even where it is data) flags the whole scan for the host."""
    lines = _bad_line_corpus()
    data = b"\n".join(lines) + b"\n"
    for cr_is_data in (False, True):
        def is_bad(l):
            return any(b >= 0x80 for b in l) or (b"\r" in l and not cr_is_data)
        exp_fb, off = [], 0
        for l in lines:
            if is_bad(l):
                exp_fb.append((off << 16) | len(l))
            off += len(l) + 1
        rest = b"".join(l + b"\n" for l in lines if not is_bad(l))
        for mode, oracle in ((dev.TOK_NONWORD_LOWER_SET, lambda d: refsem.docfreq(d)[0]),
                             (dev.TOK_NONWORD_LOWER, refsem.termfreq_nonset)):
            for chunk in (None, 4096 + 16, 100000):
                tb = ctx.textbuf(len(data) + 64)
                tb.upload_all(np.frombuffer(data, dtype=np.uint8))
                tab = ctx.table(20)
                lo = 0
                step = len(data) if chunk is None else chunk
                while lo < len(data):
                    hi = min(len(data), lo + step)
                    tab.count(tb, lo, hi, mode, cr_is_data)
                    lo = hi
                st = tab.stats()
                if text_kernel == 1:
                    assert st["flags"] & dev.TF_NONASCII and st["flags"] & dev.TF_CR and st["fallback"] == 0, st
                    tb.free()
                    tab.free()
                    continue
                assert st["flags"] == 0, st
                assert sorted(tab.fallback_lines().tolist()) == exp_fb
                codes, counts, reps = tab.fetch()
                words = keycodes.decode_table(codes, reps, mode, lambda o, n: data[o:o + n])
                got = dict(zip(words, counts.tolist()))
                if cr_is_data:
                    # '\\r' is an ordinary separator byte here (binary-mode .gz): only '\\n' ends lines
                    exp = {}
                    nl = 0
                    for l in rest.split(b"\n")[:-1]:
                        nl += 1
                        toks = refsem.RX.split(l.decode("ascii").lower())
                        for t in (set(toks) if mode == dev.TOK_NONWORD_LOWER_SET else toks):
                            exp[t] = exp.get(t, 0) + 1
                else:
                    exp = dict(oracle(rest))
                    nl = len(refsem.text_lines(rest))
                empty = exp.pop("", 0)
                assert got == exp and st["empty"] == empty and st["lines"] == nl
                tb.free()
                tab.free()


def test_fallback_list_overflow_sets_the_scan_wide_flag(ctx, text_kernel):
    """v2: more bad lines than its list holds end in the scan-wide flag; the first-generation kernel sets it for any."""
    data = "é\n".encode() * 70000      # more bad lines than the list holds (and than a warp region may isolate)
    _, st = run_count(ctx, data, dev.TOK_NONWORD_LOWER_SET, verify=False)
    assert st["flags"] & dev.TF_NONASCII


def test_upload_file_through_cufile_matches_the_ring(ctx, tmp_path):
    """The opt-in cuFile ingest (dampr_set_option("file_cufile", 1), csrc/ctx.cu): the same bytes land in the text
    buffer as through the page-locked ring; token counts agree. Skipped where cuFile is unavailable: without the
    nvidia-fs driver the upload must fail at once, naming it."""
    data = gen.text(31, 30000, V=5000)
    p = tmp_path / "c.txt"
    p.write_bytes(data)
    tb = ctx.textbuf(len(data))
    tb.set_length(len(data))
    tb.upload_file(0, str(p), 0, len(data))
    ctx.sync()
    want = tb.download(0, len(data)).tobytes()
    assert want == data
    dev.set_option("file_cufile", 1)
    try:
        tb2 = ctx.textbuf(len(data))
        tb2.set_length(len(data))
        try:
            tb2.upload_file(0, str(p), 0, len(data))
        except dev.DeviceError as e:
            assert os.path.exists("/proc/driver/nvidia-fs/version") or "nvidia-fs" in str(e), e
            if "cuFile" in str(e):
                pytest.skip("cuFile unavailable here: %s" % e)
            raise
        ctx.sync()
        assert tb2.download(0, len(data)).tobytes() == data
        # an unaligned window of the file into an unaligned offset
        tb2.upload_file(1003, str(p), 777, 50001)
        ctx.sync()
        assert tb2.download(1003, 50001).tobytes() == data[777:777 + 50001]
    finally:
        dev.set_option("file_cufile", 0)
