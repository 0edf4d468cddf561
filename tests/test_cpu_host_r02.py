"""CPU suite, round-2 additions: malformed containers, committed corpora, the numpy weight generator behind bench.py's
reference arm, and that the reference arm never loads the product library."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
from candlezip_b200 import _lib, container

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import corpus  # noqa: E402


def _var(v):
    out = bytearray()
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    out.append(v)
    return bytes(out)


def _read_gates(buf, cap):
    b = (C.c_uint8 * max(1, len(buf))).from_buffer_copy(buf or b"\0")
    rec = (C.c_uint8 * max(1, cap))()
    n = C.c_size_t(0)
    k = _lib.lib.cz_container_read_gates(b, len(buf), rec, cap, C.byref(n))
    return k, n.value, bytes(rec[:min(cap, n.value)]) if k else b""


@pytest.mark.parametrize("magic", [b"AGT2", b"AGTB"])
def test_gate_section_rejects_huge_and_truncated_counts(magic):
    """src/main.rs:2469-2484 trusts the varint count; a crafted count near 2^64 used to wrap `n + cnt` (ADVICE r1)"""
    ok = magic + _var(3) + bytes([1, 3, 5])
    k, n, rec = _read_gates(ok, 16)
    assert k == len(ok) - (2 if magic == b"AGTB" else 0) and n == 3
    for cnt in (2 ** 64 - 1, 2 ** 64 - 4, 2 ** 63, 2 ** 32, 1000):
        k, n, _ = _read_gates(magic + _var(cnt) + bytes(8), 4)
        assert k == 0, (magic, cnt)
    assert _read_gates(magic + b"\xff\xff\xff", 4)[0] == 0          # truncated varint
    assert _read_gates(magic + b"\xff" * 11 + b"\x01", 4)[0] == 0    # varint longer than 64 bits
    assert _read_gates(b"AGTX" + _var(1) + b"\0", 4)[0] == 0
    # more records than the caller's capacity: count is reported, nothing is written past `cap`
    many = magic + _var(40) + bytes(40)
    k, n, rec = _read_gates(many, 4)
    assert k and n == 40 and len(rec) == 4


def test_segment_table_and_header_reject_malformed_input():
    fields = dict(token_count=10, orig_len_bytes=10, vocab_size=256)
    blob = container.write_container(fields, b"m", [b"abc", b"defg"], seg_tokens=[6, 4])
    f, rep, gates, eng, st, pays = container.read_container(blob)
    assert pays == [b"abc", b"defg"] and list(st) == [6, 4]
    with pytest.raises(ValueError):
        container.read_container(blob[:-1])                           # byte sums larger than the file
    with pytest.raises(ValueError):
        container.read_container(blob + b"x")                         # trailing bytes the table does not account for
    hdr_len = len(container.write_container(fields, b"m", [b""]))
    seg_huge = blob[:hdr_len] + b"SEG1" + _var(2 ** 64 - 1) + _var(0) + bytes(8)
    with pytest.raises(ValueError):
        container.read_container(seg_huge)
    seg_bytes_wrap = blob[:hdr_len] + b"SEG1" + _var(2) + _var(0) + _var(5) + _var(2 ** 64 - 2) + _var(5) + _var(6) + bytes(4)
    with pytest.raises(ValueError):
        container.read_container(seg_bytes_wrap)
    bad_tokens = container.write_container(fields, b"m", [b"abc", b"defg"], seg_tokens=[6, 5])
    with pytest.raises(ValueError):
        container.read_container(bad_tokens)                          # segment tokens do not add up to token_count
    for cut in (3, 9, 11, 30, hdr_len - 1):
        with pytest.raises(ValueError):
            container.read_container(blob[:cut])                      # truncated header / repr
    # repr length pointing past the end of the file
    raw = bytearray(container.write_container(fields, b"model", [b"zz"]))
    off = raw.index(b"model") - 8
    raw[off:off + 4] = (0xFFFFFFF0).to_bytes(4, "little")
    with pytest.raises(ValueError):
        container.read_container(bytes(raw))


def test_committed_corpora_match_their_manifest():
    d = corpus.load("enwik8_3mib")
    assert len(d) == 3145728 and d[:14] == b"<mediawiki xml"
    d.decode("utf-8")
    assert len(corpus.load("alice29.txt")) == 148481 and len(corpus.load("asyoulik.txt")) == 125179
    for v in (49152, 65536):
        m = corpus.spread_map(v)
        assert len(set(m.tolist())) == 256 and m.max() < v
        ids = corpus.byte_ids(d[:70000], v, True)
        assert corpus.ids_to_bytes(ids, v, True) == d[:70000]
        assert 0.05 < ids.mean() / v < 0.2       # like the shipped SmolLM2 id traces (0.08-0.11), unlike id = byte (0.002)
    assert corpus.low_entropy_stream(100)[:27] == b"abcdefghijklmnopqrstuvwxyza" and len(corpus.low_entropy_stream(50000)) == 50000
    assert corpus.high_entropy_stream(64) == corpus.high_entropy_stream(64) and len(set(corpus.high_entropy_stream(4096))) == 256
    r = corpus.replay("alice29")
    assert len(r["proof_rows"]) == 81 and r["proof_header"][11:14] == ["gate", "candidate_id", "budget_id"] and len(r["agent_cache"]) == 43


def test_numpy_weight_generator_equals_the_products():
    """bench.py --impl reference builds its weights with tests/oracle_weights.py so that it never loads the product library;
    the two generators must agree bit for bit (counter hash, sum of four uniforms, bf16 rounding)"""
    import oracle_weights as ow

    host = cz.Context(-1)
    m = cz.Model(host, cz.SMOLLM_TINY).random_init(5, 0.05, 0.2)
    want = m.tensors()
    got = ow.smollm_random_init(cz.SMOLLM_TINY, 5, 0.05, 0.2)
    assert set(want) == set(got)
    for k in want:
        assert np.array_equal(want[k].view(np.uint32), got[k].view(np.uint32)), k
    # full-size shapes: one projection and a slice of the embedding
    big = cz.Model(host, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    for name, n in (("model.layers.17.mlp.down_proj.weight", 576 * 1536), ("model.embed_tokens.weight", 49152 * 576)):
        a = big.get_tensor(name, n)
        b = ow.tensor(name, n, 0, 0.02)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), name
    for k in ("vocab", "d_model", "n_layers", "n_heads", "n_kv_heads", "head_dim", "d_ffn", "rope_theta"):
        assert ow.SMOLLM_135M[k] == cz.SMOLLM_135M[k], k


def test_reference_arm_does_not_load_the_product_library():
    """bench.py --impl reference must run the CPU oracle alone (VERDICT r1: the ratio is void if the product .so is in that process)"""
    src = open(os.path.join(ROOT, "bench.py")).read()
    ref = src[src.index("def run_reference"):src.index("def schedule_work")] + src[src.index("class OracleSmolLM"):src.index("def run_reference")]
    assert "candlezip_b200" not in re.sub(r"#.*", "", ref)
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '0', '--warmup', '0'];\n"
            "try:\n    runpy.run_path('bench.py', run_name='__main__')\nexcept ZeroDivisionError:\n    pass\n"
            "print('LOADED', sorted({l.split()[-1].split('/')[-1] for l in open('/proc/self/maps') if 'libcandlezip' in l or 'libcz_oracle' in l}))")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert "LOADED ['libcz_oracle.so']" in r.stdout, (r.stdout[-300:], r.stderr[-300:])


def test_built_library_is_made_of_tcgen05_tma_and_fp64_kernels():
    """The hot kernels are what DESIGN.md says they are, checked on the built sm_100a SASS (cuobjdump needs no GPU): the GEMM and the
    attention kernel issue tcgen05.mma (UTCHMMA) with tensor-memory loads / stores (LDTM / STTM) and TMA (UTMALDG / UTMASTG); the
    attention kernel writes P to tensor memory (STTM); the CDF stats kernel is fed by TMA and does its arithmetic in FP64 without
    F2F conversions in the hot variants; nothing on the default path is an mma.sync (HMMA) kernel except the bisecting fallback."""
    import collections
    import re
    import shutil
    import subprocess

    if not shutil.which("cuobjdump") or not shutil.which("c++filt"):
        pytest.skip("cuobjdump / c++filt not available")
    so = os.path.join(ROOT, "candlezip_b200", "libcandlezip_b200.so")
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, timeout=300).stdout
    counts, cur = {}, None
    for line in sass.split("\n"):
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,5}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur:
            counts[cur][m.group(1)] += 1
    names = list(counts)
    dm = dict(zip(names, subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")))

    def kernels(sub):
        return [counts[n] for n in names if sub in dm[n]]

    gemm, attn = kernels("gemm_tc_kernel<"), kernels("attn_tc_kernel<")
    assert gemm and attn
    for c in gemm:
        assert c["UTCHMMA"] > 0 and c["LDTM"] > 0 and c["UTMALDG"] > 0 and c["HMMA"] == 0
    assert any(c["UTMASTG"] > 0 for c in gemm) and any(c["UTMAREDG"] > 0 for c in gemm)
    for c in attn:
        assert c["UTCHMMA"] > 0 and c["LDTM"] > 0 and c["STTM"] > 0 and c["UTMALDG"] > 0 and c["HMMA"] == 0
    stats = kernels("cdf_stats_tma_kernel<")
    assert stats and all(c["UTMALDG"] > 0 and c["DFMA"] > 0 and c["DADD"] > 0 for c in stats)
    prefix = kernels("cdf_bounds_warp_kernel<")
    assert prefix and all(c["DADD"] >= 32 for c in prefix)
    assert kernels("attn_mma_kernel<") and all(c["HMMA"] > 0 for c in kernels("attn_mma_kernel<"))  # the bisecting fallback, and only it


def test_bench_dump_outputs_is_exact_bounded_and_repeatable(tmp_path):
    """bench.py --dump-outputs: bytes as float32 and 64-bit offsets as float64 without loss, and an output over the size budget
    replaced by the same sample of its elements on every run"""
    import bench

    pay = np.random.default_rng(3).integers(0, 256, 5000).astype(np.uint8)
    off = np.array([0, 17, 2 ** 40 + 1], np.uint64)
    bench.dump_outputs(str(tmp_path / "a"), {"payload": pay, "seg_off": off})
    a, o = np.load(tmp_path / "a" / "payload.npy"), np.load(tmp_path / "a" / "seg_off.npy")
    assert a.dtype == np.float32 and np.array_equal(a, pay) and o.dtype == np.float64 and np.array_equal(o.astype(np.uint64), off)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"payload": pay, "seg_off": off}, budget=8000)
    b, c = np.load(tmp_path / "b" / "payload.npy"), np.load(tmp_path / "c" / "payload.npy")
    assert b.nbytes == 4000 and np.array_equal(b, c) and set(b.tolist()) <= set(pay.tolist())
