"""The gate's host side on RWKV-7 (whole-history rule, shared XE jobs) and the CLI's argument checks for `--backend rwkv7
--reuse-scan-dir`; no GPU needed."""
import hashlib

import numpy as np
import pytest

from candlezip_b200 import __main__ as cli
from candlezip_b200 import gate

TEXTS = {1: "Alpha Beta 12 gamma " * 9, 2: "", 3: "Delta 7 Epsilon\nno digits here " * 30, 4: "Zeta", 6: "x" * 3000}


def _tok(text, mx):
    return np.array([(ord(c) * 7) % 320 for c in text][:mx], np.uint32)


def _ids(n=1700, seed=3):
    return np.random.default_rng(seed).integers(0, 320, n).astype(np.uint32)


def _fake_bits(jobs):
    """a deterministic stand-in for cz_xe_bits: a function of (prime, targets) only"""
    out = []
    for prime, targets in jobs:
        h = hashlib.blake2b(np.asarray(prime, np.uint32).tobytes() + b"|" + np.asarray(targets, np.uint32).tobytes(), digest_size=8)
        out.append(1000.0 + int.from_bytes(h.digest(), "little") % 100000 / 100.0)
    return np.array(out)


def test_rwkv7_planning_uses_the_whole_history_and_hint():
    ids = _ids()
    seq = np.concatenate([[0], ids]).astype(np.uint32)
    big = gate.MAX_CTX_RWKV7
    jobs, plan = gate.plan_scan(ids, TEXTS, _tok, agent_chunk=256, scan_lookahead=200, max_ctx=big)
    assert [e["i"] for e in plan] == [255, 511, 767, 1023, 1279, 1535]
    for e in plan:
        i = e["i"]
        prime, targets = jobs[e["job0"]]
        assert np.array_equal(prime, seq[:i]) and np.array_equal(targets, seq[i:i + 200])
        for cid in range(4):
            h = e["hints"][cid]
            slots = e["slots"][cid * 4:cid * 4 + 4]
            if len(h) == 0:
                assert slots == [None] * 4
                continue
            assert len(set(slots)) == 1  # every budget covers the whole hint: one shared job
            assert np.array_equal(jobs[slots[0]][0], np.concatenate([seq[:i], h]))
    # decisions: the event is the whole hint after the whole history (hist_take = i + 1, BOS included)
    bits = _fake_bits(jobs)
    records, events, rows = gate.decide(plan, bits, 200, max_ctx=big)
    gated = [e for e, r in zip(plan, records) if r & 1]
    assert len(events) == len(gated) > 0
    for (i, hint, hold, ht), e, r in zip(events, gated, [r for r in records if r & 1]):
        assert i == e["i"] and ht == i + 1 and hold == i + 200
        assert np.array_equal(hint, e["hints"][(r >> 1) & 3])
    hints = [e["hints"] for e in plan]
    dec = gate.events_from_records(records, hints, 256, len(ids), scan_lookahead=200, max_ctx=big)
    assert len(dec) == len(events) and all(a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:] for a, b in zip(dec, events))
    decisions = {e["chunk_index"]: (r & 1, (r >> 1) & 3, (r >> 3) & 3) for e, r in zip(plan, records)}
    rec2, ev2 = gate.events_from_decisions(ids, TEXTS, decisions, _tok, 256, scan_lookahead=200, max_ctx=big)
    assert rec2 == records and len(ev2) == len(events)
    assert all(a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:] for a, b in zip(ev2, events))


@pytest.mark.parametrize("max_ctx", [gate.MAX_CTX_RWKV7, gate.MAX_CTX_SMOLLM])
def test_job_sharing_keeps_the_decisions(max_ctx):
    ids = _ids()
    shared, plan_s = gate.plan_scan(ids, TEXTS, _tok, 256, 200, max_ctx=max_ctx, share_jobs=True)
    every, plan_e = gate.plan_scan(ids, TEXTS, _tok, 256, 200, max_ctx=max_ctx, share_jobs=False)
    assert len(shared) < len(every)
    a = gate.decide(plan_s, _fake_bits(shared), 200, max_ctx=max_ctx)
    b = gate.decide(plan_e, _fake_bits(every), 200, max_ctx=max_ctx)
    assert a[0] == b[0] and a[2] == b[2]
    assert len(a[1]) == len(b[1]) and all(x[0] == y[0] and np.array_equal(x[1], y[1]) and x[2:] == y[2:] for x, y in zip(a[1], b[1]))


def test_smollm_job_list_is_unchanged():
    """SmolLM: one stream per non-empty (candidate, budget), in order, even where two budgets give the same prime (a short hint)"""
    ids = _ids()
    seq = np.concatenate([[0], ids]).astype(np.uint32)
    jobs, plan = gate.plan_scan(ids, TEXTS, _tok, 256, 200)
    assert gate.plan_scan(ids, TEXTS, _tok, 256, 200, max_ctx=gate.MAX_CTX_SMOLLM, share_jobs=False)[0].__len__() == len(jobs)
    bud = gate.budgets(gate.MAX_CTX_SMOLLM)
    k = 0
    for e in plan:
        i = e["i"]
        hist = seq[max(0, i - min(511, i)):i]
        assert e["job0"] == k and np.array_equal(jobs[k][0], gate.xe_prime(hist, None))
        k += 1
        for cid in range(4):
            for bid in range(4):
                h = e["hints"][cid][:bud[bid]]
                if len(h) == 0:
                    assert e["slots"][cid * 4 + bid] is None
                    continue
                assert e["slots"][cid * 4 + bid] == k and np.array_equal(jobs[k][0], gate.xe_prime(hist, h))
                k += 1
    assert k == len(jobs)
    short = plan[3]  # "Zeta": shorter than every budget, so the four budgets repeat one prime in four jobs
    assert len(set(short["slots"][:4])) == 4


def test_cli_accepts_rwkv7_gate_replay_and_refuses_segments(tmp_path, capsys):
    src = tmp_path / "in.txt"
    src.write_bytes(b"hello world " * 50)
    rdir = tmp_path / "run"
    rdir.mkdir()
    with pytest.raises(SystemExit) as e:
        cli.main(["self-test", str(src), "--backend", "rwkv7", "--reuse-scan-dir", str(rdir), "--segments", "2"])
    assert e.value.code == 2 and "--segments 1" in capsys.readouterr().err
    # accepted: the run stops later, where the (absent) device is opened, not at the argument check
    with pytest.raises(Exception) as e:
        cli.main(["self-test", str(src), "--backend", "rwkv7", "--reuse-scan-dir", str(rdir), "--device", "4096"])
    assert not isinstance(e.value, SystemExit), e.value
    assert "--reuse-scan-dir" not in capsys.readouterr().err
