"""Per-stream fault isolation and verify on the CPU: the host emulation of fab_decode_isolated / fab_verify
(tests/hostsim/hostsim.cpp) on the streams of tests/flac_corpus.py.

* every bad corpus case, placed between two good streams of the same stream_size and channel count in one buffer,
  reports [0, !=0, 0]; the good rows are bit-exact and the bad row is zero -- once more under AddressSanitizer + UBSan;
* every valid case reports all-zero status and decodes exactly, storing and not storing, by the same decoder path
  (streams walked + 1000 * frames left to the general decoder) as the plain throughput decode;
* which bit: ERROR_DECODE_INIT for unusable metadata, ERROR_DECODE_PROCESS for bad frames;
* slices examine only the frames they overlap.
"""
import functools
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

INIT, PROCESS = 1 << 13, 1 << 14
_MODE2_MAX_FRAMES = 4096      # as in test_conformance.py: longer cases are checked through their windows only
_BAD = FC.invalid_cases() + FC.damage_cases()


def _ids(cases):
    return [c.name for c in cases]


@pytest.fixture(scope="module")
def HI():
    import hostsim

    hostsim.lib()
    return hostsim


@functools.lru_cache(maxsize=None)
def good_streams(stream_size, nch):
    """Two good streams of this shape written by the library's encoder (faB2 frame tables), and what they decode to."""
    import hostsim

    rng = np.random.default_rng(stream_size * 3 + nch)
    x = np.cumsum(rng.integers(-500, 501, (2, stream_size)), axis=1)
    x = x.astype(np.int64 if nch == 2 else np.int32)
    if nch == 2:
        x = x * 977 + (x << 33)           # both words busy
    comp, st, nb, _, _ = hostsim.encode(x, level=5)
    return [bytes(comp[s:s + n]) for s, n in zip(st, nb)], x


def sandwich(bad_stream, stream_size, nch):
    """[good, bad, good] back to back in one buffer: (compressed, starts, nbytes, expected good rows)."""
    (g0, g1), x = good_streams(stream_size, nch)
    parts = [g0, bad_stream, g1]
    starts = np.cumsum([0] + [len(p) for p in parts[:-1]]).astype(np.int64)
    nbytes = np.array([len(p) for p in parts], np.int64)
    return np.frombuffer(b"".join(parts), np.uint8).copy(), starts, nbytes, x


def _frames(case):
    return sum(len(f) for f in case.frames) if case.frames else 0


# ---- bad streams between good ones -------------------------------------------------------------------------------

@pytest.mark.parametrize("case", _BAD, ids=_ids(_BAD))
def test_bad_case_isolated(HI, case):
    comp, st, nb, x = sandwich(case.streams[0], case.stream_size, case.nch)
    y, status, _ = HI.decode_isolated(comp, st, nb, case.stream_size, is_int64=case.is_int64)
    assert status[0] == 0 and status[2] == 0 and status[1] != 0, (case.name, status)
    assert np.array_equal(y[0], x[0]) and np.array_equal(y[2], x[1]), case.name
    assert not y[1].any(), case.name
    vs, _ = HI.verify(comp, st, nb, case.stream_size, is_int64=case.is_int64)
    assert np.array_equal(vs, status), (case.name, vs, status)


def test_bad_cases_isolated_under_address_and_ub_sanitizers(HI, tmp_path):
    """The [good, bad, good] calls once more, storing and not storing, against an ASan + UBSan build of the emulator in a
    child process: every read of bad input stays inside the buffers, and every status comes out the same."""
    env = HI.sanitizer_env()
    if env is None:
        pytest.skip("libasan / libubsan not available")
    so = str(tmp_path / "libhostsim_asan.so")
    HI.build(so, HI.SANITIZE)
    # the good streams come from the (unsanitised) encoder emulation in this process
    inputs = tmp_path / "inputs.npz"
    arrs = {}
    for i, case in enumerate(_BAD):
        comp, st, nb, x = sandwich(case.streams[0], case.stream_size, case.nch)
        arrs[f"c{i}"], arrs[f"s{i}"], arrs[f"n{i}"] = comp, st, nb
        arrs[f"g{i}"] = np.stack([x[0], x[1]])
        arrs[f"z{i}"] = np.array([case.stream_size, int(case.is_int64)], np.int64)
    np.savez(inputs, **arrs)
    script = textwrap.dedent(f"""
        import sys
        import numpy as np
        sys.path[:0] = [{os.path.join(HERE, "hostsim")!r}]
        import hostsim as HI
        HI.lib({so!r})
        d = np.load({str(inputs)!r})
        ok = 0
        for i in range({len(_BAD)}):
            n, i64 = (int(v) for v in d[f"z{{i}}"])
            comp, st, nb, g = d[f"c{{i}}"], d[f"s{{i}}"], d[f"n{{i}}"], d[f"g{{i}}"]
            y, s, _ = HI.decode_isolated(comp, st, nb, n, is_int64=bool(i64))
            vs, _ = HI.verify(comp, st, nb, n, is_int64=bool(i64))
            good = (s[0] == 0 and s[2] == 0 and s[1] != 0 and np.array_equal(vs, s) and np.array_equal(y[0], g[0])
                    and np.array_equal(y[2], g[1]) and not y[1].any())
            if good:
                ok += 1
            else:
                print("wrong:", i, s, vs)
        print("isolated", ok)
    """)
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-4000:]
    assert "ERROR: AddressSanitizer" not in out and "runtime error" not in out, out[-4000:]
    assert f"isolated {len(_BAD)}" in r.stdout, out[-4000:]


# ---- valid streams -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", FC.valid_cases(), ids=_ids(FC.valid_cases()))
def test_valid_case_isolated_and_verified(HI, case):
    comp, st, nb = case.buffer()
    k = len(case.streams)
    for i, (s, a, b) in enumerate(case.windows):
        y, status, _ = HI.decode_isolated(comp, st, nb, case.stream_size, a, b, is_int64=case.is_int64)
        assert not status.any(), (case.name, (s, a, b), status)
        assert np.array_equal(y[s], case.window_expect(i)), (case.name, (s, a, b))
    if case.full and _frames(case) <= _MODE2_MAX_FRAMES:
        y, status, info = HI.decode_isolated(comp, st, nb, case.stream_size, is_int64=case.is_int64)
        assert np.array_equal(status, np.zeros(k, np.int32)), (case.name, status)
        assert np.array_equal(y, case.expect), case.name
        assert info == case.info, (case.name, case.path, info)
        vs, vinfo = HI.verify(comp, st, nb, case.stream_size, is_int64=case.is_int64)
        assert np.array_equal(vs, np.zeros(k, np.int32)), (case.name, vs)
        # the no-store decoder reaches every decision by the same path as the storing one
        assert vinfo == case.info, (case.name, case.path, vinfo)


# ---- which bit ---------------------------------------------------------------------------------------------------

def _one_bad(HI, bad, stream_size=3 * FC.BS, nch=1):
    comp, st, nb, x = sandwich(bad, stream_size, nch)
    y, status, _ = HI.decode_isolated(comp, st, nb, stream_size, is_int64=nch == 2)
    vs, _ = HI.verify(comp, st, nb, stream_size, is_int64=nch == 2)
    assert np.array_equal(vs, status)
    assert np.array_equal(y[0], x[0]) and np.array_equal(y[2], x[1]) and not y[1].any()
    return int(status[1]), status


def test_init_bit_for_a_stream_cut_to_ten_bytes(HI):
    (g, _), _ = good_streams(3 * FC.BS, 1)
    bit, status = _one_bad(HI, g[:10])
    assert bit == INIT, status


def test_init_bit_for_a_bad_magic(HI):
    (g, _), _ = good_streams(3 * FC.BS, 1)
    bit, status = _one_bad(HI, b"fLaD" + g[4:])
    assert bit == INIT, status


def test_init_bit_for_a_mono_stream_in_a_stereo_call(HI):
    (mono, _), _ = good_streams(3 * FC.BS, 1)
    bit, status = _one_bad(HI, mono, nch=2)
    assert bit == INIT, status


@pytest.mark.parametrize("case", _BAD, ids=_ids(_BAD))
def test_process_bit_for_bad_frames(HI, case):
    # every invalid / damaged corpus stream has valid metadata and bad frames
    comp, st, nb, _ = sandwich(case.streams[0], case.stream_size, case.nch)
    _, status, _ = HI.decode_isolated(comp, st, nb, case.stream_size, is_int64=case.is_int64)
    assert status[1] == PROCESS, (case.name, status)


# ---- slices ------------------------------------------------------------------------------------------------------

def _four_frames_frame1_damaged():
    from oracle import flac_writer as W

    rng = np.random.default_rng(77)
    x = FC.walk(rng, 4 * FC.BS, 300)
    frs = [W.Frame(x[j * FC.BS:(j + 1) * FC.BS], [FC.sub_fixed(x[j * FC.BS:(j + 1) * FC.BS], 2, porder=2)])
           for j in range(4)]
    data, fb = W.write_stream(frs, 1)
    first = len(data) - sum(len(f) for f in fb)
    b = bytearray(data)
    b[first + len(fb[0]) + len(fb[1]) // 2] ^= 0x10          # inside the residuals of frame 1
    return bytes(b), x.astype(np.int32)


def test_slices_examine_only_their_frames(HI):
    bad, x = _four_frames_frame1_damaged()
    comp = np.frombuffer(bad, np.uint8).copy()
    st, nb = np.array([0], np.int64), np.array([len(bad)], np.int64)
    n = 4 * FC.BS
    for a, b in ((3 * FC.BS + 10, 3 * FC.BS + 100), (3 * FC.BS, n), (5, FC.BS - 1)):
        y, status, _ = HI.decode_isolated(comp, st, nb, n, a, b)
        assert status[0] == 0, (a, b, status)
        assert np.array_equal(y[0], x[a:b]), (a, b)
    for a, b in ((FC.BS - 5, FC.BS + 5), (FC.BS + 100, FC.BS + 200), (0, n), (FC.BS + 10, 3 * FC.BS + 10)):
        y, status, _ = HI.decode_isolated(comp, st, nb, n, a, b)
        assert status[0] == PROCESS, (a, b, status)
        assert not y.any(), (a, b)
    vs, _ = HI.verify(comp, st, nb, n)
    assert vs[0] == PROCESS


def test_call_level_errors_still_raise(HI):
    (g, _), _ = good_streams(3 * FC.BS, 1)
    comp = np.frombuffer(g, np.uint8).copy()
    with pytest.raises(RuntimeError, match="Decoding failed, return code = 131072"):
        HI.decode_isolated(comp, [0], [len(g)], 3 * FC.BS, 10, 3 * FC.BS + 1)
