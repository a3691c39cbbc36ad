"""Decoder conformance on the CPU: the streams of tests/flac_corpus.py (written syntax element by syntax element by
oracle/flac_writer.py) through the host emulation of the kernel bodies (tests/hostsim).

* the writer checks itself against two independent decoders (the oracle, FFmpeg);
* every valid case decodes bit-exactly in hostsim modes 0 (parallel path), 1 (walker) and 2 (throughput path: tile
  decoder + CRC pass + general decoder + walker) and through the per-stream window decode;
* mode 2 reaches the path the case was built for: `info` = streams walked + 1000 * frames left to the general decoder.
  A tile-path bug that changes a frame's length fails the chain check and the walker then returns correct samples:
  only this count shows it;
* every invalid or damaged stream fails in every mode, and once more under AddressSanitizer + UBSan, which is how an
  out-of-bounds read on bad input shows up on the CPU.
"""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "hostsim"))
sys.path.insert(0, HERE)

import flac_corpus as FC  # noqa: E402

# cases whose full decode in the emulated throughput path costs too many emulated warps: windows only
_MODE2_MAX_FRAMES = 4096


def _ids(cases):
    return [c.name for c in cases]


@pytest.fixture(scope="module")
def H():
    import hostsim

    hostsim.lib()
    return hostsim


def _frames(case):
    return sum(len(f) for f in case.frames) if case.frames else 0


def _check_windows_single(H, case, comp, st, nb, mode):
    for i, (s, a, b) in enumerate(case.windows):
        y, _ = H.decode(comp, st, nb, case.stream_size, a, b, is_int64=case.is_int64, mode=mode)
        assert np.array_equal(y[s], case.window_expect(i)), (case.name, mode, (s, a, b))


# ---- the writer against independent decoders ----------------------------------------------------------------------

def test_writer_self_check_oracle(oracle):
    for case in FC.valid_cases():
        comp, st, nb = case.buffer()
        for s in range(len(case.streams)):
            buf = comp[st[s]:st[s] + nb[s]]
            if case.full:
                y = oracle.decode_stream(buf, case.stream_size, case.nch)
                got = y.reshape(-1).view(np.int64) if case.nch == 2 else y[:, 0]
                assert np.array_equal(got, case.expect[s]), case.name
        for i, (s, a, b) in enumerate(case.windows):
            y = oracle.decode_stream(comp[st[s]:st[s] + nb[s]], case.stream_size, case.nch, a, b - a)
            got = y.reshape(-1).view(np.int64) if case.nch == 2 else y[:, 0]
            assert np.array_equal(got, case.window_expect(i)), (case.name, i)
    for case in FC.invalid_cases() + FC.damage_cases():
        with pytest.raises(RuntimeError):
            oracle.decode_stream(np.frombuffer(case.streams[0], np.uint8), case.stream_size, case.nch)


def test_writer_self_check_ffmpeg():
    from oracle import ffmpeg_flac as ff

    if not ff.available():
        pytest.skip("bundled FFmpeg FLAC codec unavailable")
    checked = 0
    for case in FC.valid_cases():
        if not (case.ffmpeg and case.full):
            continue
        for s, fb in enumerate(case.frames):
            y = ff.decode_frames(fb, case.nch)
            got = y.reshape(-1).view(np.int64) if case.nch == 2 else y[:, 0]
            assert np.array_equal(got, case.expect[s]), (case.name, s)
            checked += 1
    assert checked > 40


def test_writer_refuses_what_it_cannot_write():
    from oracle import flac_writer as W

    x = np.zeros(64, np.int64)
    x[3] = 2 ** 31
    with pytest.raises(AssertionError):          # residual of magnitude 2^31
        W.write_frame(W.Frame(x, [W.Sub("fixed", order=0, rice=W.Rice(1, 0, [30]))], number=0))
    y = np.zeros(64, np.int64)
    y[10] = 2 ** 16
    with pytest.raises(AssertionError):          # escape too narrow for its partition
        W.write_frame(W.Frame(y, [W.Sub("fixed", order=0, rice=W.Rice(0, 0, [("esc", 17)]))], number=0))
    assert W.utf8_number(0x7F) == b"\x7f" and W.utf8_number(0x80) == b"\xc2\x80"
    assert W.utf8_number(0xFFFF) == b"\xef\xbf\xbf" and len(W.utf8_number(0x10000)) == 4
    assert len(W.utf8_number(2 ** 26)) == 6 and W.utf8_number(2 ** 35)[0] == 0xFE
    assert W.crc8(b"123456789") == 0xF4 and W.crc16(b"123456789") == 0xFEE8


# ---- valid cases through the emulated decoder ---------------------------------------------------------------------

@pytest.mark.parametrize("case", FC.valid_cases(), ids=_ids(FC.valid_cases()))
def test_valid_case_hostsim(H, case):
    comp, st, nb = case.buffer()
    n = case.stream_size
    if case.full:
        for mode in (0, 1):
            y, walked = H.decode(comp, st, nb, n, is_int64=case.is_int64, mode=mode)
            assert np.array_equal(y, case.expect), (case.name, mode)
            if mode == 1:
                assert walked == len(case.streams)
    for mode in (0, 1, 2):
        _check_windows_single(H, case, comp, st, nb, mode)
    if case.full and _frames(case) <= _MODE2_MAX_FRAMES:
        y, info = H.decode(comp, st, nb, n, is_int64=case.is_int64, mode=2)
        assert np.array_equal(y, case.expect), case.name
        assert info == case.info, (case.name, case.path, info)
        if case.path == "tile":
            assert info == 0
        elif case.path == "general":
            assert info > 0 and info % 1000 == 0
        else:
            assert info % 1000 > 0


@pytest.mark.parametrize("case", FC.valid_cases(), ids=_ids(FC.valid_cases()))
def test_valid_case_hostsim_windows(H, case):
    comp, st, nb = case.buffer()
    ws = np.array([w[0] for w in case.windows], np.int64)
    wf = np.array([w[1] for w in case.windows], np.int64)
    wl = np.array([w[2] for w in case.windows], np.int64)
    data, offs, _ = H.decode_windows(comp, st, nb, case.stream_size, ws, wf, wl, is_int64=case.is_int64, bsh=case.hint())
    for i in range(ws.size):
        assert np.array_equal(data[offs[i]:offs[i + 1]], case.window_expect(i)), (case.name, case.windows[i])
    if case.full and _frames(case) <= _MODE2_MAX_FRAMES:
        k = len(case.streams)
        data, offs, _ = H.decode_windows(comp, st, nb, case.stream_size, np.arange(k), np.zeros(k, np.int64),
                                         np.full(k, case.stream_size), is_int64=case.is_int64, bsh=case.hint())
        assert np.array_equal(data.reshape(k, -1), case.expect), case.name


# ---- stage 1: the product's warp body against the serial reference -------------------------------------------------

_ALL = FC.valid_cases() + FC.invalid_cases() + FC.damage_cases()


def _library_case(H):
    """Three streams of the library's own encoder (emulated): frame-size tables of 81 frames, so that the warp scan
    carries its offset across three 32-frame chunks."""
    rng = np.random.default_rng(5)
    x = np.cumsum(rng.integers(-500, 501, (3, 80 * 1152 + 5)), axis=1).astype(np.int32)
    comp, st, nb, _, _ = H.encode(x, level=0)
    return FC.Case("library_encoded_81_frames", [bytes(comp[s:s + n]) for s, n in zip(st, nb)], x.shape[1], 1)


@pytest.mark.parametrize("case", _ALL + (None,), ids=_ids(_ALL) + ["library_encoded_81_frames"])
def test_meta_warp_body_matches_meta_body(H, case):
    """k_dec_meta's warp body (lane 0 parses, the warp scans the frame-size table) and meta_body agree on the metadata,
    the frame offsets, the stream flags and the status, with the call's channel count and with the other one (which
    makes every stream undecodable)."""
    case = case or _library_case(H)
    comp, st, nb = case.buffer()
    for nch in (case.nch, 3 - case.nch):
        want = H.meta(comp, st, nb, case.stream_size, nch, warp=False)
        got = H.meta(comp, st, nb, case.stream_size, nch, warp=True)
        for name, g, w in zip(("meta", "frame offsets", "stream flags", "status"), got, want):
            assert np.array_equal(g, w), (case.name, nch, name)
        assert ((want[2] == 4) == (want[3] != 0)).all() and (nch == case.nch or (want[2] == 4).all()), case.name


# ---- bad input -----------------------------------------------------------------------------------------------------

_BAD = FC.invalid_cases() + FC.damage_cases()


@pytest.mark.parametrize("case", _BAD, ids=_ids(_BAD))
def test_bad_case_raises(H, case):
    comp, st, nb = case.buffer()
    for mode in (0, 1, 2):
        with pytest.raises(RuntimeError, match="Decoding failed"):
            H.decode(comp, st, nb, case.stream_size, is_int64=case.is_int64, mode=mode)
    with pytest.raises(RuntimeError, match="Decoding failed"):
        H.decode_windows(comp, st, nb, case.stream_size, [0], [0], [case.stream_size], is_int64=case.is_int64,
                         bsh=case.hint())


def test_bad_cases_under_address_and_ub_sanitizers(H, tmp_path):
    """The invalid and damaged streams once more, against an ASan + UBSan build of the emulator in a child process:
    every read the kernel bodies make of bad input must stay inside the buffers (the decode must still fail)."""
    env = H.sanitizer_env()
    if env is None:
        pytest.skip("libasan / libubsan not available")
    so = str(tmp_path / "libhostsim_asan.so")
    H.build(so, H.SANITIZE)
    script = textwrap.dedent(f"""
        import sys
        sys.path[:0] = [{os.path.join(HERE, "hostsim")!r}, {HERE!r}, {os.path.dirname(HERE)!r}]
        import hostsim
        import flac_corpus as FC
        hostsim.lib({so!r})
        n = 0
        for case in FC.invalid_cases() + FC.damage_cases():
            comp, st, nb = case.buffer()
            for mode in (0, 1, 2):
                try:
                    hostsim.decode(comp, st, nb, case.stream_size, is_int64=case.is_int64, mode=mode)
                except RuntimeError:
                    n += 1
                else:
                    print("no error:", case.name, mode)
        print("raised", n)
    """)
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-4000:]
    assert "ERROR: AddressSanitizer" not in out and "runtime error" not in out, out[-4000:]
    assert f"raised {3 * len(_BAD)}" in r.stdout, out[-4000:]
