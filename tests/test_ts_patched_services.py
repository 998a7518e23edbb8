"""The TypeScript drop-in, executed: a senweaver-ide checkout with ts/patches/*.ed applied is run end to end on the CPU
(oracle/ts_harness/run_patched.py) — the PATCHED `_computeRewardSignals`, `_refreshEngineStats`, `getStats`, `_buildReport`,
`_analyzePatterns` and the functions of ts/traceRecordCodec.ts, unmodified, in the in-repo TypeScript-subset interpreter, with
`IApoScoringService` answered by byte blocks in the C ABI's formats (computed by the oracle; in the IDE: by the B200 engine).
Everything they return must equal what the UNPATCHED reference returned for the same inputs (tests/golden/ref_*.json, the parity
pin): the per-trace reward dimensions and finalReward bit for bit, the whole PromptEffectivenessReport object (tallies, per-mode
stats in first-appearance order, the six patterns with ids / severities / example previews, the dimension-low patterns, every
generated suggestion), and the collector / APO stats.  Those tests need the senweaver-ide checkout (the patches apply to it;
its source is not part of this repository, see run_reference.CHECKOUT).  The micro-batching test of ts/apoScoringMainService.ts
needs only this repository."""
import json
import math
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle", "ts_harness"))
import run_reference as rr  # noqa: E402

REF = rr.CHECKOUT
needs_checkout = pytest.mark.skipif(not os.path.exists(os.path.join(REF, rr.APO_REL)),
                                    reason="needs the senweaver-ide checkout (SENWEAVER_IDE_CHECKOUT)")


def num(v):
    """fixture number: binary64 as a hex string, JS integer literals as JSON integers"""
    if isinstance(v, str) and (v == "nan" or v.lstrip("-").startswith("0x")):
        return math.nan if v == "nan" else float.fromhex(v)
    return v


def same(a, b, tol=0.0, path=""):
    """deep equality; numbers by value (0 == 0.0: one JS Number), optionally within a relative tolerance"""
    a, b = num(a), num(b)
    if isinstance(a, bool) or isinstance(b, bool) or a is None or b is None or isinstance(a, str) or isinstance(b, str):
        assert a == b and type(a) is type(b), (path, a, b)
    elif isinstance(a, (int, float)) and isinstance(b, (int, float)):
        if isinstance(a, float) and math.isnan(a):
            assert isinstance(b, float) and math.isnan(b), (path, a, b)
        else:
            assert a == b or (tol and abs(a - b) <= tol * max(1.0, abs(a), abs(b))), (path, a, b)
    elif isinstance(a, dict):
        assert isinstance(b, dict) and list(a) == list(b), (path, list(a), list(b) if isinstance(b, dict) else b)      # key ORDER too
        for k in a:
            same(a[k], b[k], tol, f"{path}/{k}")
    else:
        assert isinstance(a, list) and isinstance(b, list) and len(a) == len(b), (path, a, b)
        for i, (x, y) in enumerate(zip(a, b)):
            same(x, y, tol, f"{path}[{i}]")


@pytest.fixture(scope="module")
def outputs(orc):
    sys.path.insert(0, os.path.join(ROOT, "oracle", "ts_harness"))
    import run_patched as rp
    return rp.build_outputs(REF)


@needs_checkout
def test_the_patched_methods_are_the_ones_that_ran(outputs):
    _, _, calls, lines = outputs
    assert calls["rewardBatch"] > 431 and calls["score"] > 11          # every reward and every report went through the service
    sys.path.insert(0, os.path.join(ROOT, "ts", "patches"))
    import make_patches as mp
    tcs, apo = mp.patched_text(REF, mp.TCS).split("\n"), mp.patched_text(REF, mp.APO).split("\n")
    for key, text in (("TCS._computeRewardSignals", tcs), ("TCS._refreshEngineStats", tcs), ("APO._buildReport", apo)):
        a, b = lines[key]
        assert "this._scoring." in "\n".join(text[a - 1:b]), key
    a, b = lines["APO._analyzePatterns"]
    assert "R.patterns.forEach" in "\n".join(apo[a - 1:b])


@needs_checkout
def test_patched_reward_signals_equal_the_reference_bit_for_bit(outputs):
    cases = outputs[0]
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_reward_cases.json")))["cases"]
    assert len(cases) == len(want) == 431
    for c, w in zip(cases, want):
        assert c["name"] == w["name"] and c["dims"] == w["dims"] and c["finalReward"] == w["finalReward"], c["name"]


@needs_checkout
def test_patched_reports_and_stats_equal_the_reference(outputs):
    reports = outputs[1]
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_report_cases.json")))["corpora"]
    assert set(reports) == set(want) and len(reports) == 11
    for cname, got in reports.items():
        w = want[cname]
        same(got["report"], w["report"], 0.0, f"{cname}/report")               # the object APOService returns: exact
        # what _buildReport hands to _generateLocalSuggestions: the engine's sums are exact integers / 2^52, the reference adds
        # doubles in trace order -> equal to ~1e-15 relative, and equal in everything derived from them above
        same(got["locals"], w["locals"], 1e-12, f"{cname}/locals")
        same(got["stats"], w["stats"], 1e-12, f"{cname}/stats")


@needs_checkout
def test_patched_evaluate_beam_feeds_the_strict_greater_adoption(orc):
    """`_evaluateBeam` (new) + `_applyBeamUpdate` (the reference's inline bookkeeping of APO:1138-1166, moved into a method by the
    patch): scores and top-K come back as little-endian blocks, the beam is the candidates in top-K order with their scores, a new
    best is adopted only on a strictly greater score, the round counter advances per evaluation."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle", "ts_harness"))
    import run_patched as rp
    P = rp.Patched(REF)
    C, T = 6, 300
    dims = orc.gen_dims(0x5EED00B7, 0, C, 0, T, 300, 2)
    scores, _ = orc.score_dims(dims)
    order = [int(c) for c in orc.topk(scores, 4)]
    cands = [{"id": f"p{c}", "version": c + 1, "content": f"prompt {c}"} for c in range(C)]
    st = P.evaluate_beam(cands, dims)
    assert [b["id"] for b in st["beam"]] == [f"p{c}" for c in order]                        # K = min(beamWidth 4, C)
    assert [b["score"] for b in st["beam"]] == [float(scores[c]) for c in order] and st["beam"][0]["content"] == f"prompt {order[0]}"
    assert st["currentRound"] == 1 and st["totalRounds"] == 3 and st["historyBestScore"] == float(scores[order[0]])
    assert st["historyBestPrompt"]["id"] == f"p{order[0]}" and [a["id"] for a in P.adopted] == [f"p{order[0]}"]
    st = P.evaluate_beam(cands, dims)                                                         # same scores again: not strictly greater
    assert st["currentRound"] == 2 and len(P.adopted) == 1
    worse = dims.copy()
    worse[order[0]] = -1.0                                                                    # the former best drops to the bottom
    st = P.evaluate_beam(cands, worse)
    assert st["currentRound"] == 3 and len(P.adopted) == 1 and st["beam"][0]["id"] == f"p{order[1]}"
    assert st["historyBestPrompt"]["id"] == f"p{order[0]}"                                   # history keeps the best ever seen
    better = dims.copy()
    better[order[3]] = 1.0
    st = P.evaluate_beam(cands, better)
    assert [a["id"] for a in P.adopted] == [f"p{order[0]}", f"p{order[3]}"] and st["historyBestScore"] == 1.0
    assert P.evaluate_beam([], dims[:0]) == st                                                # no candidates: nothing happens


def test_main_service_micro_batches_single_trace_rewards(orc):
    """ts/apoScoringMainService.ts `_flushRewards`, executed: the single-trace reward requests of one tick are concatenated into ONE
    addon call and the three result blocks are sliced back per caller (72 / 4 / 8 bytes per record) — each caller must receive exactly
    what a call of its own would have returned, whatever the mix of request sizes."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle", "ts_harness"))
    import minijs as js
    import run_patched as rp
    import run_reference as rr
    src = open(os.path.join(ROOT, "ts", "apoScoringMainService.ts"), encoding="utf-8").read()
    text, _ = rr.extract_method(src, "_flushRewards")
    interp = js.Interp({"Uint8Array": js.NativeFunction(rp.uint8array), "RECORD_BYTES": 32,
                        "VSBuffer": js.JSObject(wrap=js.NativeFunction(lambda this, u8: js.JSObject(buffer=u8)))})
    scoring = rp.OracleScoring()
    seen = []

    def addon_reward_batch(this, handle, array_buffer):
        assert isinstance(array_buffer, rp.ByteBuf) and handle == "H"
        seen.append(len(array_buffer.b) // 32)
        r = scoring.reward_batch(None, js.JSObject(buffer=rp.uint8array(None, array_buffer))).value
        # the addon hands back plain ArrayBuffers
        return js.SyncPromise(js.JSObject(dims=r["dims"]["buffer"]["buffer"], masks=r["masks"]["buffer"]["buffer"], finals=r["finals"]["buffer"]["buffer"]))

    recs = orc.gen_records(0x5EED00C3, orc.STREAM_CORPUS, 0, 1, 0, 11, 400, 1).reshape(-1)
    sizes = [1, 3, 1, 2, 4]                                           # five callers in one tick
    got, chunks, at = {}, [], 0
    this = js.JSObject(_addon=js.JSObject(rewardBatch=js.NativeFunction(addon_reward_batch)), _handle="H", _pendingRewards=js.JSArray())
    for k, n in enumerate(sizes):
        chunk = recs[at:at + n]
        at += n
        chunks.append(chunk)
        u8 = rp.uint8array(None, rp.ByteBuf(b"\xEE" * 5 + chunk.tobytes() + b"\xEE" * 3), 5, 32 * n)        # a view into a larger buffer
        this["_pendingRewards"].append(js.JSObject(records=u8, resolve=js.NativeFunction(lambda t, v, k=k: got.__setitem__(k, v)),
                                                   reject=js.NativeFunction(lambda t, e: (_ for _ in ()).throw(AssertionError(e)))))
    _, fn = interp.make_method(text, this)
    interp.call(fn, this, [])
    assert seen == [sum(sizes)] and len(this["_pendingRewards"]) == 0 and sorted(got) == list(range(len(sizes)))
    for k, chunk in enumerate(chunks):
        want = scoring.reward_batch(None, rp.vsbuffer(chunk.tobytes())).value
        for block in ("dims", "masks", "finals"):
            assert rp.vsbuffer_bytes(got[k][block]) == rp.vsbuffer_bytes(want[block]), (k, block)
    interp.call(fn, this, [])                                          # nothing pending: no call
    assert seen == [sum(sizes)]
