"""The reference-side TypeScript binding (ts/patches/*.ed + the three new files in ts/) keeps the service surface byte for byte
(SURVEY 8b).  Always: the edit commands of the committed ed scripts stay clear of the interface / decorator / registration
lines.  With the reference checkout present: the scripts apply (patch --ed), reproduce what ts/patches/make_patches.py
generates, leave `ITraceCollectorService` (TCS:133-210), `IAPOService` (APO:203-267), the decorator ids (TCS:212, APO:269),
the exported types, the storage keys and both `registerSingleton(..., Delayed)` lines untouched, and the four reductions
(`_computeRewardSignals`, `getStats`, `_buildReport`, `_analyzePatterns`) delegate to IApoScoringService."""
import hashlib
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATCHES = os.path.join(ROOT, "ts", "patches")
sys.path.insert(0, PATCHES)
import make_patches as mp  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "oracle", "ts_harness"))
import run_reference as rr  # noqa: E402

REF = rr.CHECKOUT
REF_PRESENT = os.path.exists(os.path.join(REF, mp.TCS))
# 1-based inclusive line ranges of the reference that no patch may touch
PROTECTED = {
    mp.TCS: [(17, 212, "exported types + ITraceCollectorService + decorator id"), (216, 217, "storage keys"), (969, 969, "registerSingleton")],
    mp.APO: [(19, 269, "exported types + IAPOService + decorator id"), (273, 275, "storage keys"), (1545, 1545, "registerSingleton")],
}


def ed_commands(path):
    """[(first, last, op)] of an ed script produced by `diff -e`."""
    cmds, in_text = [], False
    for ln in open(path, encoding="utf-8").read().split("\n"):
        if in_text:
            if ln == ".":
                in_text = False
            continue
        m = re.fullmatch(r"(\d+)(?:,(\d+))?([acd])", ln)
        if m:
            a, b, op = int(m.group(1)), int(m.group(2) or m.group(1)), m.group(3)
            cmds.append((a, b, op))
            in_text = op in "ac"
    return cmds


@pytest.mark.parametrize("rel,_fn,out", mp.TARGETS)
def test_patches_stay_clear_of_the_service_surface(rel, _fn, out):
    cmds = ed_commands(os.path.join(PATCHES, out))
    assert cmds, out
    base = open(os.path.join(PATCHES, out + ".base")).read().split()
    assert base[0] == rel and base[1] == "sha256" and len(base[2]) == 64
    for first, last, op in cmds:
        for lo, hi, what in PROTECTED.get(rel, []):
            if op == "a":
                assert not (lo <= first < hi), (out, first, what)        # appending after the LAST protected line is fine
            else:
                assert last < lo or first > hi, (out, first, last, what)


def test_new_ts_files_declare_the_channel_and_the_codec():
    svc = open(os.path.join(ROOT, "ts", "apoScoringService.ts")).read()
    main = open(os.path.join(ROOT, "ts", "apoScoringMainService.ts")).read()
    codec = open(os.path.join(ROOT, "ts", "traceRecordCodec.ts")).read()
    assert "createDecorator<IApoScoringService>('senweaverApoScoringService')" in svc and "registerSingleton(IApoScoringService, ApoScoringService, InstantiationType.Delayed)" in svc
    for m in ("rewardBatch", "dimsUpload", "rolloutsUpload", "corpusUpload", "scoreResident", "score", "scoreHostRecords"):
        assert re.search(r"\b" + m + r"\(", svc) and re.search(r"async " + m + r"\(", main), m
    assert "queueMicrotask(() => this._flushRewards())" in main                # single-trace calls of one tick are coalesced
    assert "export const EMPTY_DIMS" in codec and "export function decodeCorpusReport" in codec


@pytest.mark.skipif(not REF_PRESENT, reason="needs the senweaver-ide checkout (SENWEAVER_IDE_CHECKOUT)")
@pytest.mark.parametrize("rel,_fn,out", mp.TARGETS)
def test_patches_apply_and_keep_the_interfaces_byte_for_byte(tmp_path, rel, _fn, out):
    src = os.path.join(REF, rel)
    sha = open(os.path.join(PATCHES, out + ".base")).read().split()[2]
    assert hashlib.sha256(open(src, "rb").read()).hexdigest() == sha
    work = tmp_path / os.path.basename(rel)
    shutil.copy(src, work)
    os.chmod(work, 0o644)
    r = subprocess.run([sys.executable, os.path.join(PATCHES, "make_patches.py"), "--apply", os.path.join(PATCHES, out), str(work)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    got = open(work, encoding="utf-8").read()
    assert got == mp.patched_text(REF, rel)                                        # the committed script is what the generator emits
    ref_lines = open(src, encoding="utf-8").read().split("\n")
    for lo, hi, what in PROTECTED.get(rel, []):
        block = "\n".join(ref_lines[lo - 1:hi])
        assert block in got, what
    if rel == mp.TCS:
        assert ref_lines[132].startswith("export interface ITraceCollectorService") and ref_lines[211].startswith("export const ITraceCollectorService = createDecorator")
        assert "senweaverTraceCollectorService" in ref_lines[211]
        body = got[got.index("private _computeRewardSignals("):got.index("// --- Backend Upload (required for Phase 2 training) ---", got.index("private _computeRewardSignals("))]
        assert "this._scoring.rewardBatch(" in body and "weightedSum" not in body and "toolSuccessRate * 2 - 1" not in body
        g0 = got.index("\tgetStats(): TraceCollectorStats {")
        stats = got[g0:got.index("\tgetAllTraces(): ConversationTrace[] {", g0)]
        assert "this._engineStats" in stats and "rewardSum +=" not in stats
        assert got.count("@IApoScoringService private readonly _scoring: IApoScoringService,") == 1
        # injection order of the existing dependencies is unchanged: the new one comes last
        ctor = got[got.index("\tconstructor("):got.index("\t) {", got.index("\tconstructor("))]
        order = [ctor.index(k) for k in ("@IStorageService", "@IProductService", "@IRequestService", "@IApoScoringService")]
        assert order == sorted(order)
    if rel == mp.APO:
        assert ref_lines[202].startswith("export interface IAPOService") and "senweaverAPOService" in ref_lines[268]
        rep = got[got.index("private async _buildReport("):got.index("\tprivate _extractMode(")]
        assert "await this._scoring.score(" in rep and ".reduce(" not in rep and "goodCount++" not in rep
        pat = got[got.index("\tprivate _analyzePatterns(R: CorpusReportNumbers"):got.index("\tprivate _generateLocalSuggestions(")]
        assert "traces.filter(" not in pat and "R.patterns.forEach" in pat
        assert "const report = await this._buildReport(traces);" in got
        assert "private async _evaluateBeam(" in got and "this._applyBeamUpdate(serverResponse.beamUpdate);" in got
        assert "bu.bestScore > this._beamState.historyBestScore" in got           # the strict '>' adoption is still the reference's
        ctor = got[got.index("\tconstructor("):got.index("\t) {", got.index("\tconstructor("))]
        order = [ctor.index(k) for k in ("@IStorageService", "@IProductService", "@IRequestService", "@ITraceCollectorService", "@IApoScoringService")]
        assert order == sorted(order)
    if rel == mp.APP:
        assert "services.set(IApoScoringService, new SyncDescriptor(ApoScoringMainService, undefined, false));" in got
        assert "mainProcessElectronServer.registerChannel(APO_SCORING_CHANNEL, apoScoringChannel);" in got
