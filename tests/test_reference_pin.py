"""THE PARITY PIN (SURVEY 8c).  tests/golden/ref_*.json hold outputs of the reference's OWN functions —
`_computeRewardSignals`, `getStats` (traceCollectorService.ts), `_buildReport`, `_analyzePatterns`, `_generateLocalSuggestions`,
`getStats` (apoService.ts) — produced by executing their unmodified source text (oracle/ts_harness/run_reference.py: extracted
from the reference checkout at generation time, run by the minijs interpreter; run_reference.mjs does the same under Node).

  * not gpu: the C oracle and the Python transcription reproduce every reference value bit for bit (409 traces: the SURVEY
    KATs, seeded random traces, every threshold hit exactly in both modes; 11 corpora incl. the no-bad early-out, unscored
    traces and the empty corpus); when the reference checkout is present, the committed fixtures are re-derived from it and
    must be identical; the interpreter's own semantics are pinned by known JavaScript results.
  * gpu: the CUDA engine (apo_reward_batch, the corpus scan + report) reproduces the same reference values through the C ABI.
"""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "oracle", "ts_harness")
sys.path.insert(0, HARNESS)
import run_reference as rr  # noqa: E402
from oracle import ts_transcription as ts  # noqa: E402

REF = rr.CHECKOUT
REF_PRESENT = os.path.exists(os.path.join(REF, rr.TCS_REL))
DIMS = ts.DIM_ORDER
PAT_DESCR = [
    "Users give negative feedback after errors occur in conversations",
    "Tool call failures lead to user dissatisfaction",
    "User feedback is poor in conversations with high token consumption",
    "Users still dissatisfied after multiple LLM calls (possible retries)",
    "Long conversations with many turns still result in user dissatisfaction",
    "Slow tool execution (>15s total) correlates with user dissatisfaction",
]
SEV = {"low": 0, "medium": 1, "high": 2}
MODE_CODE = {"unknown": 0, "normal": 1, "agent": 2, "gather": 3, "designer": 4}


def unhex(v):
    """Fixture number -> float: binary64 values are hex strings, JS integer literals (`goodRate : 0`) stay JSON integers."""
    if v is None:
        return None
    if isinstance(v, (int, float)):
        return float(v)
    return math.nan if v == "nan" else float.fromhex(v)


def same_bits(a, b):
    return (math.isnan(a) and math.isnan(b)) or (a == b and math.copysign(1, a) == math.copysign(1, b))


@pytest.fixture(scope="module")
def ref_reward():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "ref_reward_cases.json")))


@pytest.fixture(scope="module")
def ref_report():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "ref_report_cases.json")))


def record_of(tup, scored=True):
    t = ts.make_trace(*tup)
    if scored:
        ts.compute_reward_signals(t)
    return np.frombuffer(ts.encode_record(t), dtype=np.dtype([("raw", "V32")]))[0], t


def test_fixtures_come_from_the_reference_text(ref_reward, ref_report):
    prov = ref_reward["provenance"]
    assert "unmodified reference method text" in prov["engine"] or prov["engine"].startswith("node")
    assert prov["method_lines"]["TCS._computeRewardSignals"] == [668, 788]          # SURVEY 8a row a3/a4
    assert prov["method_lines"]["APO._buildReport"] == [498, 625] and prov["method_lines"]["APO._analyzePatterns"] == [635, 773]
    assert len(ref_reward["cases"]) >= 400 and len(ref_report["corpora"]) >= 10
    if not REF_PRESENT:
        return
    import hashlib
    for rel, sha in prov["reference"].items():                                     # the very files they were generated from
        assert hashlib.sha256(open(os.path.join(REF, rel), "rb").read()).hexdigest() == sha
    r = subprocess.run([sys.executable, os.path.join(HARNESS, "run_reference.py"), "--reference", REF, "--check"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.count("identical to what the reference text produces") == 3, r.stdout + r.stderr


def test_kats_of_the_survey_are_what_the_reference_computes(ref_reward):
    by = {c["name"]: c for c in ref_reward["cases"]}
    want = {"K1": 1.0, "K2": -0.43600000000000005, "K3": -0.21700000000000003, "K4": 0.20930232558139533, "K5": 0.639,
            "K6": -0.2542857142857143, "K7": 0.05157894736842105}
    for k, v in want.items():
        assert unhex(by[k]["finalReward"]) == v, k


def test_c_oracle_and_transcription_match_the_reference_per_trace(orc, ref_reward):
    for c in ref_reward["cases"]:
        tup = tuple(c["input"])
        rec, t = record_of(tup)
        want = {d["name"]: unhex(d["value"]) for d in c["dims"]}
        # the independent Python transcription, on the reference's object shape
        got_t = {d["name"]: d["value"] for d in t["summary"]["rewardDimensions"]}
        assert list(got_t) == [d["name"] for d in c["dims"]], c["name"]            # same dims pushed, same order
        assert all(same_bits(float(got_t[n]), want[n]) for n in want), c["name"]
        assert same_bits(float(t["summary"]["finalReward"]), unhex(c["finalReward"])), c["name"]
        # the C oracle, on the packed record
        d, mask, fr = orc.reward_one(np.frombuffer(rec.tobytes(), orc.RECORD_DTYPE))
        for i, n in enumerate(DIMS):
            assert bool(mask >> i & 1) == (n in want), (c["name"], n)
            if n in want:
                assert same_bits(float(d[i]), want[n]), (c["name"], n, d[i], want[n])
        assert same_bits(float(fr), unhex(c["finalReward"])), c["name"]


def corpus_records(orc, cname, idx):
    traces = rr.corpus_traces(cname, idx)
    for t in traces:
        if t.get("_score", True):
            ts.compute_reward_signals(t)
    raw = b"".join(ts.encode_record(t) for t in traces)
    return np.frombuffer(raw, orc.RECORD_DTYPE).copy(), traces


def check_report_against_reference(rep, ref, idx, exact_means):
    """rep: a report struct of the C oracle or the engine (same field names); ref: one corpus of ref_report_cases.json."""
    R, L = ref["report"], ref["locals"]
    assert (rep.total, rep.good, rep.bad, rep.none) == (R["totalConversations"], R["goodFeedbackCount"], R["badFeedbackCount"], R["noFeedbackCount"])
    assert same_bits(rep.goodRate, unhex(R["goodRate"]))
    for mode, st in R["byMode"].items():
        m = MODE_CODE[mode]
        assert list(rep.byMode[m]) == [st["total"], st["good"], st["bad"]], mode
        assert same_bits(rep.byModeGoodRate[m], unhex(st["goodRate"])), mode
    assert sum(int(rep.byMode[m][0]) for m in range(5)) == R["totalConversations"]
    close = (lambda a, b: same_bits(a, b)) if exact_means else (lambda a, b: abs(a - b) <= 1e-12 * max(1.0, abs(b)))
    if L.get("avgReward") is None:
        assert rep.withReward == 0 and math.isnan(rep.avgReward)
    else:
        assert close(rep.avgReward, unhex(L["avgReward"]))
    rbd = L.get("rewardByDimension") or {}
    for i, n in enumerate(DIMS):
        if n in rbd:
            assert rep.dim[i].count == rbd[n]["count"], n
            assert close(rep.dim[i].sum, unhex(rbd[n]["sum"])) and close(rep.dim[i].avg, unhex(rbd[n]["avg"])), n
        else:
            assert rep.dim[i].count == 0, n
    # the six problem patterns: emitted ones carry frequency / severity / first-3 examples; absent ones are below their minimum
    emitted = {p["description"]: p for p in R["patterns"]}
    for p, descr in enumerate(PAT_DESCR):
        if descr in emitted:
            e = emitted[descr]
            assert rep.pat[p].flag == 1 and rep.pat[p].count == e["frequency"] and rep.pat[p].severity == SEV[e["severity"]], descr
            want_idx = [int(x["threadId"].split("-")[1]) for x in e["examples"]]
            got_idx = [idx[k] for k in rep.pat[p].examples if k >= 0]
            assert got_idx == want_idx, descr
        else:
            assert rep.pat[p].flag == 0, descr
    # dim-low patterns (APO:574-596) and dimension suggestions (APO:800-827) are derived rules: flags and severities
    low = {p["description"].split(" dimension")[0]: p for p in R["patterns"] if "dimension reward signal consistently low" in p["description"]}
    sugg = {s["description"].split(" dimension")[0]: s for s in R["suggestions"] if "dimension performing poorly" in s["description"]}
    for i, n in enumerate(DIMS):
        assert bool(rep.dim[i].low_flag) == (n in low), n
        if n in low:
            assert rep.dim[i].low_severity == SEV[low[n]["severity"]] and rep.dim[i].count == low[n]["frequency"]
        assert bool(rep.dim[i].sugg_flag) == (n in sugg), n
        if n in sugg:
            assert rep.dim[i].sugg_priority == SEV[sugg[n]["priority"]]
    S = ref["stats"]["traceCollector"]
    assert (rep.toolCalls, rep.toolSucc, rep.toolFail) == (S["totalToolCalls"], S["totalToolSucceeded"], S["totalToolFailed"])
    if S["toolSuccessRate"] is None:
        assert math.isnan(rep.toolSuccessRate)
    else:
        assert same_bits(rep.toolSuccessRate, unhex(S["toolSuccessRate"]))
    assert rep.withReward == S["tracesWithReward"]
    if S["avgFinalReward"] is not None:
        assert close(rep.avgReward, unhex(S["avgFinalReward"]))                   # TCS.getStats and APO._buildReport take the same mean


def test_c_oracle_report_matches_the_reference_build_report(orc, ref_report):
    for cname, ref in ref_report["corpora"].items():
        recs, _ = corpus_records(orc, cname, ref["indices"])
        rep = orc.report(recs) if len(recs) else orc.report(np.zeros(0, orc.RECORD_DTYPE))
        check_report_against_reference(rep, ref, ref["indices"], exact_means=True)    # sequential binary64 sums: the same bits


def test_transcription_report_matches_the_reference(ref_report):
    for cname, ref in ref_report["corpora"].items():
        traces = rr.corpus_traces(cname, ref["indices"])
        for t in traces:
            if t.get("_score", True):
                ts.compute_reward_signals(t)
        rep = ts.build_report(traces)
        R, L = ref["report"], ref["locals"]
        assert (rep["goodFeedbackCount"], rep["badFeedbackCount"], rep["noFeedbackCount"]) == (R["goodFeedbackCount"], R["badFeedbackCount"], R["noFeedbackCount"])
        assert (rep["avgReward"] is None) == (L.get("avgReward") is None)
        if rep["avgReward"] is not None:
            assert same_bits(float(rep["avgReward"]), unhex(L["avgReward"])), cname
        assert [p["frequency"] for p in rep["patterns"]] == [p["frequency"] for p in R["patterns"] if p["description"] in PAT_DESCR]


def test_apo_getstats_recent_mean_is_reproduced(ref_report):
    """APOService.getStats: mean finalReward of the 20 most recent traces (stable sort by startTime desc, APO:1478-1487)."""
    for cname, ref in ref_report["corpora"].items():
        traces = rr.corpus_traces(cname, ref["indices"])
        for t in traces:
            if t.get("_score", True):
                ts.compute_reward_signals(t)
        scored = [t for t in traces if t["summary"]["finalReward"] is not None]
        recent = sorted(scored, key=lambda t: -t["startTime"])[:20]              # Python's sort is stable, like Array.prototype.sort
        want = ref["stats"]["apo"]["avgFinalReward"]
        if not recent:
            assert want is None
            continue
        acc = 0
        for t in recent:
            acc = acc + (t["summary"]["finalReward"] or 0)
        assert same_bits(acc / len(recent), unhex(want)), cname


# ------------------------------------------------------------------------------------------------ the interpreter itself
def test_minijs_semantics_known_javascript_results():
    import minijs as js
    I = js.Interp()

    def run(src, **vars_):
        env = js.Env(I.g)
        env.vars.update({k: js.to_js(v) for k, v in vars_.items()})
        return js.from_js(I.ev_top(js.Parser(src).expression(), env, js.undefined))

    assert run("0.1 + 0.2") == 0.30000000000000004
    assert run("1 - 3 * 0.4") == -0.20000000000000018                       # K2's response_efficiency term
    assert run("(2.5).toFixed(0)") == "3" and run("(0.125).toFixed(2)") == "0.13" and run("(1.005).toFixed(2)") == "1.00"
    assert run("(-0.0004).toFixed(3)") == "-0.000" and run("(12.3456).toFixed(1)") == "12.3" and run("(0.5).toFixed(0)") == "1"
    assert run("a?.b.c || 'x'", a=None) == "x" and run("a?.b.c || 'x'", a={"b": {"c": "y"}}) == "y"
    assert run("a.b ?? 5", a={}) == 5 and run("a.b ?? 5", a={"b": 0}) == 0 and run("a.b || 5", a={"b": 0}) == 5
    assert run("Math.max(-1, 1 - Math.max(0, n - 1) * 0.4)", n=7) == -1 and run("Math.min(3, 2)") == 2
    assert run("x === 'good' ? 1.0 : x === 'bad' ? -1.0 : 0.0", x="bad") == -1.0
    assert run("[3,1,2].filter(v => v > 1).map(v => v * 2).reduce((s, v) => s + v, 0)") == 10
    assert run("[{k:2,i:0},{k:1,i:1},{k:2,i:2},{k:1,i:3}].sort((a, b) => b.k - a.k).map(o => o.i)") == [0, 2, 1, 3]   # stable
    assert run("`n=${n} avg: ${v.toFixed(3)}`", n=4, v=-0.30049) == "n=4 avg: -0.300"
    assert run("1 / 0") == math.inf and math.isnan(run("0 / 0")) and run("'a' + 1 + 2") == "a12" and run("1 + 2 + 'a'") == "3a"
    assert run("Object.entries(o).map(([k, v]) => k + v)", o={"b": 1, "a": 2}) == ["b1", "a2"]                        # insertion order
    assert run("null === undefined") is False and run("x !== null", x=None) is False and run("typeof y", y=1.5) == "number"
    assert run("s.substring(0, 3)", s="abcdef") == "abc" and run("[1,2,3,4].slice(0, 3)") == [1, 2, 3]
    # constructs the codec / the patched services add (tests/test_ts_codec.py, tests/test_ts_patched_services.py)
    assert run("0x80 | (d > 0 ? 0x04 : 0) | (d > 15000 ? 0x08 : 0)", d=20000.5) == 0x8C and run("(m >> 2) & 1", m=0b1101) == 1
    assert run("1 << 31") == -2147483648 and run("(1 << 31) >>> 0") == 2147483648 and run("5 ^ 3") == 6 and run("-1 >>> 28") == 15
    assert run("a | b === 1", a=2, b=1) == 3 and run("(4294967296 + 7) | 0") == 7 and run("x instanceof y", x=1, y=2) is False
    assert run("await p", p=js.SyncPromise(41)) == 41 and run("await 5") == 5
    assert run("p.then(v => v + 1).then(v => v * 2)", p=js.SyncPromise(20)).value == 42
    assert run("p.then(v => v + 1).catch(e => 'caught ' + e)", p=js.SyncPromise(error="boom", rejected=True)).value == "caught boom"
    name, fn = I.make_method("f(a: number, b = a * 2, c: string = 'z'): string { return a + b + c; }", js.undefined)
    assert I.call(fn, js.undefined, [1]) == "3z" and I.call(fn, js.undefined, [1, 5, "y"]) == "6y"
    with pytest.raises(js.JSUnsupported):                    # what the interpreter does not model fails loudly instead of guessing
        run("'k' in o", o={})


# ------------------------------------------------------------------------------------------------ the CUDA engine
@pytest.mark.gpu
def test_engine_rewards_match_the_reference_bit_for_bit(engine, orc, ref_reward):
    recs = np.frombuffer(b"".join(record_of(tuple(c["input"]))[0].tobytes() for c in ref_reward["cases"]), orc.RECORD_DTYPE)
    dims, masks, finals = engine.reward_batch(recs)
    for k, c in enumerate(ref_reward["cases"]):
        want = {d["name"]: unhex(d["value"]) for d in c["dims"]}
        for i, n in enumerate(DIMS):
            assert bool(masks[k] >> i & 1) == (n in want), (c["name"], n)
            if n in want:
                assert same_bits(float(dims[k, i]), want[n]), (c["name"], n)
        assert same_bits(float(finals[k]), unhex(c["finalReward"])), c["name"]
    # and one at a time (the zero-copy single-trace path of endTrace / recordUserFeedback)
    for k in (0, 1, 6, 100, 300):
        d1, m1, f1 = engine.reward_batch(recs[k:k + 1])
        assert m1[0] == masks[k] and same_bits(float(f1[0]), float(finals[k]))


@pytest.mark.gpu
def test_engine_report_matches_the_reference_build_report(engine, orc, ref_report):
    for cname, ref in ref_report["corpora"].items():
        recs, _ = corpus_records(orc, cname, ref["indices"])
        if len(recs) == 0:
            continue
        engine.corpus_upload(recs)
        engine.dims_upload(np.full((1, 4, 9), np.nan, np.float32))
        for tuning in (0, 1):                               # corpus scan inside the scoring launch / stand-alone K2
            engine.set_tuning(tuning)
            rep = engine.score(1, 0, corpus=True).report
            # exact integer sums vs the reference's sequential binary64 sums: equal to ~1e-16, compared at 1e-12
            check_report_against_reference(rep, ref, ref["indices"], exact_means=False)
        engine.set_tuning(0)
