#!/usr/bin/env python
"""Runs the reference's OWN hot-path functions and writes the golden fixtures that pin the oracle.

    python oracle/ts_harness/run_reference.py [--reference /root/reference] [--check]

The reference is TypeScript and this image has no JS runtime, so the method texts are extracted from the reference checkout
at run time (by method name, balanced braces — nothing is copied into the repo) and executed UNMODIFIED by
oracle/ts_harness/minijs.py, a small interpreter for the TypeScript subset they use.  Executed methods:

    traceCollectorService.ts : _computeRewardSignals, getStats
    apoService.ts            : _buildReport, _extractMode, _analyzePatterns, _generateLocalSuggestions, getStats

Inputs are the 12-tuples of tests/golden/make_golden.py (the SURVEY 8c KATs + seeded random traces, built as
ConversationTrace objects in the reference's own shape).  Outputs: tests/golden/ref_reward_cases.json and
tests/golden/ref_report_cases.json with binary64 values as hex strings and a provenance block (engine, sha256 of the two
reference files, line ranges of the extracted methods).  tests/test_reference_pin.py holds the C oracle, the Python
transcription and (-m gpu) the CUDA engine to these values bit for bit, and — when the reference checkout is present —
re-runs this script in --check mode to prove the committed fixtures are what the reference text produces.

oracle/ts_harness/run_reference.mjs does the same under Node >= 18 (type stripping + `new Function`), for any machine that
has one: identical fixture format, engine "node".
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import minijs as js  # noqa: E402

TCS_REL = "src/vs/workbench/contrib/senweaver/common/traceCollectorService.ts"
APO_REL = "src/vs/workbench/contrib/senweaver/common/apoService.ts"
GOLDEN = os.path.join(ROOT, "tests", "golden")
# The senweaver-ide checkout the fixtures and ts/patches were generated against (its source is never copied into this
# repository); SENWEAVER_IDE_CHECKOUT names another.  The tests that need it skip where it is absent.
CHECKOUT = os.environ.get("SENWEAVER_IDE_CHECKOUT", "/root/reference")


# ------------------------------------------------------------------------------------------------ method extraction
def extract_method(text: str, name: str):
    """Source text and 1-based line range of the class method `name` (declaration at one tab of indentation)."""
    import re
    m, i, j = None, 0, 0
    for cand in re.finditer(r"^\t(?:(?:private|public|protected)\s+)?(?:async\s+)?" + re.escape(name) + r"\s*\(", text, re.M):
        i = text.index("(", cand.start())
        depth = 0
        while True:                                   # parameter list: balanced parentheses
            c = text[i]
            if c == "(":
                depth += 1
            elif c == ")":
                depth -= 1
                if depth == 0:
                    break
            i += 1
        # a class method has a body: the first '{' outside the return-type annotation's <...> comes before any ';'
        # (the same name inside the service interface is a signature ending in ';')
        j, adepth, body = i + 1, 0, False
        while j < len(text):
            c = text[j]
            if c in "<[(":
                adepth += 1
            elif c in ">])":
                adepth -= 1
            elif c == ";" and adepth == 0:
                break
            elif c == "{" and adepth == 0:
                body = True
                break
            j += 1
        if body:
            m = cand
            break
    if m is None:
        raise KeyError(name)
    k, depth = j, 0
    in_str = None
    while True:
        c = text[k]
        if in_str:
            if c == "\\":
                k += 1
            elif c == in_str:
                in_str = None
            elif in_str == "`" and text.startswith("${", k):
                # template expression: skip to its closing brace (no nested templates in these methods)
                d2, k = 1, k + 2
                while d2:
                    if text[k] == "{":
                        d2 += 1
                    elif text[k] == "}":
                        d2 -= 1
                    k += 1
                continue
        elif c in "'\"`":
            in_str = c
        elif text.startswith("//", k):
            k = text.index("\n", k)
            continue
        elif text.startswith("/*", k):
            k = text.index("*/", k) + 1
        elif c == "{":
            depth += 1
        elif c == "}":
            depth -= 1
            if depth == 0:
                break
        k += 1
    src = text[m.start():k + 1]
    first = text.count("\n", 0, m.start()) + 1
    return src, (first, first + src.count("\n"))


class Reference:
    def __init__(self, ref_root: str):
        self.tcs_text = open(os.path.join(ref_root, TCS_REL), encoding="utf-8").read()
        self.apo_text = open(os.path.join(ref_root, APO_REL), encoding="utf-8").read()
        self.lines = {}
        self.uuid = 0
        self.spy = {}
        glob = {
            "generateUuid": js.NativeFunction(self._uuid),
            "Date": js.JSObject(now=js.NativeFunction(lambda this: 1700000000000)),
            "console": js.JSObject(warn=js.NativeFunction(lambda this, *a: js.undefined), log=js.NativeFunction(lambda this, *a: js.undefined)),
        }
        self.interp = js.Interp(glob)
        # ---- TraceCollectorService instance state the methods touch
        self.tcs = js.JSObject(_traces=js.JSMap(), _feedbacks=js.JSMap(),
                               _estimateStorageBytes=js.NativeFunction(lambda this: 0))
        for name in ("_computeRewardSignals", "getStats"):
            self.tcs[name] = self._method(self.tcs_text, "TCS", name, self.tcs)
        # ---- APOService instance state
        self.apo = js.JSObject(_suggestions=js.JSArray(), _segments=js.JSArray(), _reports=js.JSArray(), _beamState=None,
                               _textualGradients=js.JSArray(),
                               _onDidGenerateSuggestions=js.JSObject(fire=js.NativeFunction(lambda this, *a: js.undefined)),
                               _traceCollectorService=js.JSObject(getAllTraces=js.NativeFunction(lambda this: js.JSArray(self.tcs["_traces"].d.values()))))
        for name in ("_buildReport", "_extractMode", "_analyzePatterns", "_generateLocalSuggestions", "getStats"):
            self.apo[name] = self._method(self.apo_text, "APO", name, self.apo)
        # observe the locals _buildReport hands to _generateLocalSuggestions (avgReward, rewardByDimension never leave the method otherwise)
        real = self.apo["_generateLocalSuggestions"]

        def spy(this, *args):
            self.spy = {"goodRate": args[0], "avgReward": args[3] if len(args) > 3 else js.undefined,
                        "rewardByDimension": args[4] if len(args) > 4 else js.undefined}
            return self.interp.call(real, self.apo, list(args))
        self.apo["_generateLocalSuggestions"] = js.NativeFunction(spy)

    def _uuid(self, this):
        self.uuid += 1
        return f"uuid-{self.uuid}"

    def _method(self, text, tag, name, this):
        src, rng = extract_method(text, name)
        self.lines[f"{tag}.{name}"] = list(rng)
        _, fn = self.interp.make_method(src, this)
        return fn

    # -- the calls
    def compute_reward_signals(self, trace: dict) -> dict:
        t = js.to_js(trace)
        self.interp.call(self.tcs["_computeRewardSignals"], self.tcs, [t])
        return js.from_js(t)

    def build_report(self, traces: list[dict]) -> dict:
        ts = js.JSArray(js.to_js(t) for t in traces)
        for t in ts:                                   # as endTrace / recordUserFeedback would have done (TCS:413, 547)
            if t["summary"]["finalReward"] is None and t.get("_score", True):
                self.interp.call(self.tcs["_computeRewardSignals"], self.tcs, [t])
        self.apo["_suggestions"] = js.JSArray()
        self.spy = {}
        rep = self.interp.call(self.apo["_buildReport"], self.apo, [ts])
        return {"report": js.from_js(rep), "locals": js.from_js(js.JSObject(self.spy)), "traces": js.from_js(ts)}

    def stats(self, traces: list[dict]) -> dict:
        self.tcs["_traces"] = js.JSMap((t["id"], js.to_js(t)) for t in traces)
        self.tcs["_feedbacks"] = js.JSMap((t["id"], t["summary"]["userFeedback"]) for t in traces if t["summary"]["userFeedback"])
        a = self.interp.call(self.tcs["getStats"], self.tcs, [])
        b = self.interp.call(self.apo["getStats"], self.apo, [])
        return {"traceCollector": js.from_js(a), "apo": js.from_js(b)}


# ------------------------------------------------------------------------------------------------ fixtures
def hexf(x):
    if x is None:
        return None
    if isinstance(x, bool):
        return x
    if isinstance(x, (int, float)):
        x = float(x)
        return "nan" if math.isnan(x) else x.hex()
    return x


def hexify(o):
    if isinstance(o, dict):
        return {k: hexify(v) for k, v in o.items()}
    if isinstance(o, list):
        return [hexify(v) for v in o]
    if isinstance(o, float):
        return hexf(o)
    return o


def golden_inputs():
    sys.path.insert(0, GOLDEN)
    import make_golden as mg
    rng = random.Random(0x5EED)
    tuples = [("K%d" % i, mg.KATS["K%d" % i]) for i in range(1, 8)]
    tuples += [("r%03d" % i, mg.random_tuple(rng)) for i in range(256)]
    # thresholds hit exactly (strict '>' vs '>='), both modes: the places a restatement most easily gets wrong
    edge = []
    for mode in ("normal", "agent"):
        for fail in range(0, 7):
            edge.append((None, False, True, 8, 8 - min(fail, 8), min(fail, 8), 4000, 1, 100, 1, 1, mode))
        for tc in (3, 4, 6, 7, 8, 9, 10, 11, 15, 16, 25, 26):
            edge.append((None, False, True, tc, tc, 0, 1000 * tc, 2, 2000, 2, 2, mode))
            edge.append((None, False, True, tc, tc, 0, 1000 * tc + 1, 2, 2001, 2, 2, mode))
        for dur_per in (999.5, 1000, 1000.5, 3000, 3000.25, 10000, 10000.5):
            edge.append(("bad", False, True, 3, 2, 1, dur_per * 3, 3, 5000, 3, 3, mode))
        for llm in range(0, 9):
            edge.append(("good", False, False, 0, 0, 0, 0, llm, 0, 1, llm, mode))
        for tok in (1999, 2000, 2001, 4999, 5000, 5001, 9999, 10000, 10001, 14999, 15000, 15001, 29999, 30000, 30001):
            edge.append((None, True, True, 0, 0, 0, 0, 1, tok, 1, 1, mode))
        for turns in range(0, 11):
            edge.append(("bad", False, True, 0, 0, 0, 0, 1, 0, turns, turns + 1, mode))
        # durations a binary32 copy would put on the other side of a threshold (the record's durClass carries the binary64 answer)
        for dur, calls in ((1000.00001, 1), (3000.0000001, 1), (10000.0000001, 1), (15000.0000001, 1), (15000.0004, 2), (6000.0000002, 2),
                           (29999.9999999, 3), (30000.000000001, 3), (1e-9, 4), (16777217.0, 1), (2999.99999999, 1)):
            edge.append(("bad", False, True, calls, calls, 0, dur, 2, 1500, 2, 2, mode))
    tuples += [("e%03d" % i, t) for i, t in enumerate(edge)]
    return tuples


def corpus_index() -> dict:
    """name -> indices into golden_inputs() of the traces that make up the corpus."""
    n = len(golden_inputs())
    tuples = [t for _, t in golden_inputs()]
    rng = random.Random(0x5EEDC0)
    corpora = {"all": list(range(n)), "first40": list(range(40)),
               "no_bad": [i for i, t in enumerate(tuples) if t[0] != "bad"][:60], "tiny": [0, 1, 2], "empty": []}
    for k in range(6):
        corpora[f"sample{k}"] = sorted(rng.sample(range(n), rng.choice([12, 30, 77, 150])))
    return corpora


def corpus_traces(cname: str, idx: list) -> list:
    """ConversationTrace objects (reference shape) of one corpus: ids, start times, span previews, and — in the sample
    corpora — every ninth trace left unscored (never ended, never rated: finalReward stays null, TCS:397)."""
    from oracle import ts_transcription as ts
    tuples = [t for _, t in golden_inputs()]
    traces = []
    for n, i in enumerate(idx):
        t = ts.make_trace(*tuples[i])
        t["id"], t["threadId"], t["startTime"] = f"trace-{i}", f"thread-{i}", float(1000 + (i * 7919) % 1013)
        for sp_i, sp in enumerate(t["spans"]):
            sp["data"]["contentPreview"] = f"{sp['type']} {i}.{sp_i}"
            if sp["type"] == "tool_call":
                sp["data"]["toolName"] = f"tool{sp_i % 3}"
                sp["data"]["toolResult"] = "x" * (90 + 7 * (sp_i % 4))
        if cname.startswith("sample") and n % 9 == 4:
            t["_score"] = False
        traces.append(t)
    return traces


def build_fixtures(ref_root: str):
    from oracle import ts_transcription as ts
    R = Reference(ref_root)
    prov = {
        "engine": "minijs (oracle/ts_harness/minijs.py) executing the unmodified reference method text",
        "reference": {TCS_REL: hashlib.sha256(R.tcs_text.encode()).hexdigest(), APO_REL: hashlib.sha256(R.apo_text.encode()).hexdigest()},
        "method_lines": R.lines,
    }
    cases = []
    for name, tup in golden_inputs():
        t = ts.make_trace(*tup)
        out = R.compute_reward_signals(t)
        s = out["summary"]
        cases.append({"name": name, "input": list(tup),
                      "dims": [{"name": d["name"], "value": hexf(d["value"])} for d in s["rewardDimensions"]],
                      "finalReward": hexf(s["finalReward"])})
    reward = {"provenance": prov, "cases": cases}

    # ---- corpora for _buildReport / getStats: whole set, subsets, the "no bad trace" early-out, unscored traces
    reports = {}
    for cname, idx in corpus_index().items():
        traces = corpus_traces(cname, idx)
        res = R.build_report(traces)
        res["stats"] = R.stats(res["traces"])
        res["indices"] = idx
        res["unscored"] = [n for n, t in enumerate(traces) if t.get("_score") is False]
        del res["traces"]
        reports[cname] = hexify(res)
    report = {"provenance": prov, "corpora": reports}
    return reward, report


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default=CHECKOUT)
    ap.add_argument("--check", action="store_true", help="compare with the committed fixtures instead of writing them")
    args = ap.parse_args()
    reward, report = build_fixtures(args.reference)
    # the inputs, for run_reference.mjs (Node): the same tuples, corpora and unscored markers
    inputs = {"tuples": [[n, list(t)] for n, t in golden_inputs()],
              "corpora": {c: {"indices": idx, "unscored": [n for n, t in enumerate(corpus_traces(c, idx)) if t.get("_score") is False]}
                          for c, idx in corpus_index().items()}}
    paths = {"ref_reward_cases.json": reward, "ref_report_cases.json": report, "ref_inputs.json": inputs}
    rc = 0
    for fname, obj in paths.items():
        p = os.path.join(GOLDEN, fname)
        if args.check:
            same = os.path.exists(p) and json.load(open(p)) == json.loads(json.dumps(obj))
            print(f"{fname}: {'identical to what the reference text produces' if same else 'DIFFERS'}")
            rc |= 0 if same else 1
        else:
            with open(p, "w") as f:
                json.dump(obj, f, indent=0, sort_keys=False)
            print(f"wrote {p}")
    return rc


if __name__ == "__main__":
    sys.exit(main())
