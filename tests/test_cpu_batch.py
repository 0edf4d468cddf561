"""CPU suite for the many-file codec (codec.compress_many / decompress_many): the planning with fake encode / decode calls --
segment packing, the sort permutation and its inverse, waves, grouping by decode settings, fallback selection and the per-blob
errors.  A fake model with the Model.encode / Model.decode signatures (the "payload" of a segment is its ids) runs the whole file-level
path without a GPU."""
import numpy as np
import pytest

from candlezip_b200 import _lib, codec, container, split_segments

NONE = _lib.NO_ZERO_WIDTH
ZW_TOKEN = 255  # the fake coder's zero-width token (unless coded with the floored pdf)


class FakeModel:
    """Model.encode / Model.decode stand-in: a segment's payload is b"F" (floored pdf) or b"P", then its ids as uint32.  Token
    ZW_TOKEN is zero-width without the floor.  Records every call; decode checks the lock-step precondition."""

    def __init__(self, arch=0):
        self.cfg = dict(arch=arch, vocab=256)
        self.engine = 0
        self.encodes, self.decodes = [], []

    def encode(self, ids, n_segments=1, bos=0, context=512, reprime_interval=512, seg_start=None, pdf_floor=False, zero_width_out=False):
        ids = np.asarray(ids, np.uint32)
        seg = split_segments(len(ids), n_segments) if seg_start is None else np.asarray(seg_start, np.uint64)
        self.encodes.append(dict(n_tokens=len(ids), n_segments=len(seg) - 1, pdf_floor=pdf_floor))
        pays, zw = [], np.full(len(seg) - 1, NONE, np.uint64)
        for g in range(len(seg) - 1):
            s = ids[int(seg[g]) : int(seg[g + 1])]
            hit = np.nonzero(s == ZW_TOKEN)[0]
            if hit.size and not pdf_floor:
                if not zero_width_out:
                    raise _lib.CzError(_lib.CZ_ERR_ZERO_WIDTH, f"zero-width coding interval at coded index {int(seg[g]) + int(hit[0])}")
                zw[g] = hit[0]
                pays.append(b"?")  # unspecified
                continue
            pays.append((b"F" if pdf_floor else b"P") + s.tobytes())
        return (pays, seg, zw) if zero_width_out else (pays, seg)

    def decode(self, payloads, seg_start, bos=0, context=512, reprime_interval=512, pdf_floor=False):
        seg = np.asarray(seg_start, np.uint64)
        lens = np.diff(seg)
        assert np.all(lens[:-1] >= lens[1:]), "lock-step precondition: non-increasing segment lengths"
        self.decodes.append(dict(key=(bos, context, reprime_interval, pdf_floor), n_segments=len(payloads), lens=lens.tolist()))
        out = []
        for p, n in zip(payloads, lens):
            assert p[:1] == (b"F" if pdf_floor else b"P")
            x = np.frombuffer(p[1:], np.uint32)
            assert x.shape[0] == int(n)
            out.append(x)
        return np.concatenate(out).astype(np.uint32) if out else np.zeros(0, np.uint32)


def _files(rng, lengths, avoid_zw=True):
    out = []
    for n in lengths:
        b = rng.integers(0, 255 if avoid_zw else 256, n).astype(np.uint8)
        out.append(bytes(b))
    return out


def test_pack_segments_matches_split_segments():
    lengths = [0, 5, 1, 7, 0, 3]
    for nseg in (1, 3, 8):
        seg, ranges, local = codec.pack_segments(lengths, nseg)
        assert seg[0] == 0 and int(seg[-1]) == sum(lengths) and len(ranges) == len(lengths)
        off = 0
        for n, (g0, g1), loc in zip(lengths, ranges, local):
            assert np.array_equal(loc, split_segments(n, nseg))
            assert np.array_equal(seg[g0 : g1 + 1] - off, loc)
            off += n
        assert ranges[-1][1] == len(seg) - 1


@pytest.mark.parametrize("max_streams", [1, 3, 7, 2048])
def test_unpermutation_and_waves(max_streams):
    """shuffled segment lengths, zeros included: every file gets its ids back in order; no wave exceeds max_streams and every wave is
    non-increasing"""
    rng = np.random.default_rng(max_streams)
    jobs, pays, want = [], [], []
    for f in range(23):
        lens = rng.integers(0, 9, rng.integers(1, 5)).tolist()
        if f % 5 == 0:
            lens[0] = 0
        ids = [rng.integers(0, 1000, n).astype(np.uint32) for n in lens]
        jobs.append(((0, 512, 512, False), lens))
        pays.append([x.tobytes() for x in ids])
        want.append(np.concatenate(ids).astype(np.uint32))
    calls = []

    def decode_fn(key, payloads, seg_start):
        lens = np.diff(seg_start)
        calls.append(lens)
        assert len(payloads) <= max_streams and np.all(lens[:-1] >= lens[1:]) and np.all(lens > 0)
        return np.concatenate([np.frombuffer(p, np.uint32) for p in payloads])

    got = codec.decode_many(jobs, pays, decode_fn, max_streams)
    for f in range(len(jobs)):
        assert np.array_equal(got[f], want[f]), f
    n_live = sum(1 for _, lens in jobs for n in lens if n > 0)
    assert sum(len(c) for c in calls) == n_live and len(calls) == -(-n_live // max_streams)
    waves = codec.decode_waves(jobs, max_streams)
    assert [len(w) for _, w in waves] == [len(c) for c in calls]
    with pytest.raises(ValueError):
        codec.decode_waves(jobs, 0)


def test_waves_sort_is_stable():
    jobs = [((0, 512, 512, False), [4, 2]), ((0, 512, 512, False), [4, 4, 2])]
    [(key, items)] = codec.decode_waves(jobs, 100)
    assert items == [(0, 0, 4), (1, 0, 4), (1, 1, 4), (0, 1, 2), (1, 2, 2)]


def test_different_settings_never_share_a_call():
    keys = [(0, 512, 512, False), (0, 256, 512, False), (0, 512, 256, False), (0, 512, 512, True), (7, 512, 512, False)]
    jobs = [(keys[f % len(keys)], [3, 2]) for f in range(17)]
    pays = [[bytes([f]) * 3, bytes([f]) * 2] for f in range(17)]
    seen = []

    def decode_fn(key, payloads, seg_start):
        files = {p[0] for p in payloads}
        assert all(jobs[f][0] == key for f in files), (key, files)
        seen.append(key)
        return np.concatenate([np.frombuffer(p, np.uint8).astype(np.uint32) for p in payloads])

    got = codec.decode_many(jobs, pays, decode_fn, 4)
    assert sorted(set(seen)) == sorted(keys)
    for f in range(17):
        assert got[f].tolist() == [f] * 5


def test_fallback_selection():
    ranges = [(0, 2), (2, 3), (3, 3), (3, 6)]
    zw = np.full(6, NONE, np.uint64)
    assert codec.zero_width_files(ranges, zw) == [] and codec.zero_width_files(ranges, None) == []
    zw[4] = 0
    zw[1] = 17
    assert codec.zero_width_files(ranges, zw) == [0, 3]
    # encode_many: exactly the reporting files fall back; "floor" re-codes them (and only them) in one call
    lists = [np.array([1, 2, 3, 4], np.uint32), np.array([ZW_TOKEN, 1], np.uint32), np.zeros(0, np.uint32),
             np.array([5, 6, 7, 8, 9, ZW_TOKEN], np.uint32), np.array([9], np.uint32)]
    for policy in ("stored", "floor"):
        m = FakeModel()

        def encode_fn(ids, seg, pdf_floor):
            if pdf_floor:
                return m.encode(ids, seg_start=seg, pdf_floor=True)[0], None
            return m.encode(ids, seg_start=seg, zero_width_out=True)[::2]

        res = codec.encode_many(lists, 2, encode_fn, policy)
        flags = [r[2] for r in res]
        fb = _lib.CZ_FLAG_STORED if policy == "stored" else _lib.CZ_FLAG_PDF_FLOOR
        assert flags == [0, fb, 0, fb, 0], policy
        if policy == "floor":
            assert len(m.encodes) == 2 and m.encodes[1] == dict(n_tokens=8, n_segments=4, pdf_floor=True)
            assert res[3][0] == [b"F" + lists[3][:3].tobytes(), b"F" + lists[3][3:].tobytes()]
        else:
            assert len(m.encodes) == 1 and res[1][0] is None
        assert np.array_equal(res[0][1], split_segments(4, 2)) and res[0][0] == [b"P" + lists[0][:2].tobytes(), b"P" + lists[0][2:].tobytes()]
    assert codec.encode_many([], 1, None) == []
    with pytest.raises(ValueError):
        codec.encode_many(lists, 1, None, "skip")


@pytest.mark.parametrize("policy", ["stored", "floor"])
@pytest.mark.parametrize("nseg", [1, 3])
def test_compress_many_equals_compress_and_round_trips(policy, nseg):
    rng = np.random.default_rng(nseg)
    datas = _files(rng, [0, 1, 2, 5, 40, 7, 0, 13])
    datas[3] = b"ab\xffcd"  # zero-width for the fake coder
    datas[5] = b"\xff" * 7
    m = FakeModel()
    many = codec.compress_many(m, datas, n_segments=nseg, context=256, on_zero_width=policy)
    assert len(m.encodes) == (2 if policy == "floor" else 1)
    single = [codec.compress(m, d, n_segments=nseg, context=256, on_zero_width=policy) for d in datas]
    assert many == single
    m.decodes.clear()
    assert codec.decompress_many(m, many, max_streams=2) == datas
    assert all(c["n_segments"] <= 2 for c in m.decodes)
    assert codec.decompress_many(m, many) == [codec.decompress(m, b) for b in many]


def test_stored_and_empty_make_no_call():
    m = FakeModel()
    datas = [b"", b"\xff", b"", b"x\xffy"]
    blobs = codec.compress_many(m, datas)
    flags = [container.read_container(b)[0]["reserved_flags"] for b in blobs]
    assert [bool(f & _lib.CZ_FLAG_STORED) for f in flags] == [False, True, False, True]
    m.decodes.clear()
    assert codec.decompress_many(m, blobs) == datas and m.decodes == []
    assert codec.decompress_many(m, []) == [] and codec.compress_many(m, []) == []


def test_errors_name_the_blob():
    m = FakeModel()
    datas = [b"hello", b"world!", b"abc", b"defg"]
    blobs = codec.compress_many(m, datas)
    f, rep, _, _, _, pays = container.read_container(blobs[2])
    gated = container.write_container(dict(f), rep, pays, gates=[1, 0, 1])
    with pytest.raises(ValueError, match=r"^blob 2: gated"):
        codec.decompress_many(m, blobs[:2] + [gated] + blobs[3:])
    f, rep, _, _, _, pays = container.read_container(blobs[1])
    bad = container.write_container(dict(f, orig_hash16=b"\x01" * 16), rep, pays)
    with pytest.raises(ValueError, match=r"^blob 1: decoded bytes do not match"):
        codec.decompress_many(m, [blobs[0], bad] + blobs[2:])
    assert codec.decompress_many(m, [blobs[0], bad] + blobs[2:], verify=False)[1] == datas[1]
    with pytest.raises(ValueError, match=r"^blob 3: bad container header"):
        codec.decompress_many(m, blobs[:3] + [b"\x00" * 7])
    stored = codec.compress(m, b"q\xffq")
    broken = stored[:-1] + b"Q"
    with pytest.raises(ValueError, match=r"^blob 0: stored payload"):
        codec.decompress_many(m, [broken, blobs[0]])


def test_cli_many_refuses_the_gate_replay(capsys):
    """argument checks of compress-many / decompress-many that come before any model is built"""
    from candlezip_b200.__main__ import main

    for argv in (["compress-many", "a", "b", "--reuse-scan-dir", "d"], ["decompress-many", "a", "--max-streams", "0"],
                 ["compress", "a", "b", "c"], ["decompress-many", "a", "--segments", "2"], ["decompress-many", "a", "--on-zero-width", "floor"],
                 ["compress-many", "a", "--max-streams", "8"], ["compress", "a", "--max-streams", "8"]):
        with pytest.raises(SystemExit) as e:
            main(argv)
        assert e.value.code == 2, argv
    err = capsys.readouterr().err
    assert "--reuse-scan-dir" in err and "--max-streams" in err and "INPUT [OUTPUT]" in err and "compress settings" in err
    assert "applies to decompress-many only" in err


def test_floored_call_is_checked_for_zero_width():
    """the floored re-code runs with the zero-width report too: a file reported there is an error, not a silent container"""
    lists = [np.array([1, ZW_TOKEN], np.uint32), np.array([2, 3], np.uint32)]

    def encode_fn(ids, seg, pdf_floor):
        zw = np.full(len(seg) - 1, NONE, np.uint64)
        zw[0] = 1  # the first segment of every call reports, floored or not
        return [b"x"] * (len(seg) - 1), zw

    with pytest.raises(RuntimeError, match=r"files \[0\] met a zero-width token under the floored pdf"):
        codec.encode_many(lists, 1, encode_fn, "floor")
