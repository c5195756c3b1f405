"""The C oracle against OUTPUTS OF THE REFERENCE'S OWN CODE (tests/golden/ref_js.json).

The vectors were produced in the build container by executing the reference's minified segmentor / formants / stats /
utterance modules (/root/reference/dist/main.js:2, inner modules 3/4/0/7) with oracle/minijs -- see
tests/golden/make_ref_js_golden.py.  Everything is compared exactly: seg_ci (dropped segments included), syllable tables,
Float32Array(9) formant rows (checksums), the 53-dim rows as doubles bit for bit, callback order, and the time stamps the
reference hands to its callback (numbers for levels 4/5, toFixed(3) strings for 10/13)."""
import json
import os
import sys

import numpy as np
import pytest
from conftest import GOLDEN, sha

sys.path.insert(0, GOLDEN)
import npzparts  # noqa: E402
from framegen import adversarial_frames, dropped_segment_frames, voiced_random_frames  # noqa: E402

from oracle import oracle  # noqa: E402
from oracle.minijs import Interp  # noqa: E402
from oracle.minijs import run_reference  # noqa: E402
from oracle.minijs.interp import to_str  # noqa: E402
from webspeechanalyzer_b200 import FaConfig, api, synth_speech  # noqa: E402
from webspeechanalyzer_b200.engine import UtteranceResult  # noqa: E402

DOC = json.load(open(os.path.join(GOLDEN, "ref_js.json")))
CASES = {c["name"]: c for c in DOC["cases"]}
DOC12 = json.load(open(os.path.join(GOLDEN, "ref_js_l12.json")))      # level 12 (make_coeffs / polyfit / numeric), own fixture
CASES12 = {c["name"]: c for c in DOC12["cases"]}
DOC3 = json.load(open(os.path.join(GOLDEN, "ref_js_l3.json")))        # level 3 (raw ranked tracks), own fixture
CASES3 = {c["name"]: c for c in DOC3["cases"]}
_wav = {}


def frames_for(inp, cfg):
    if inp["kind"] == "wav_full":
        if not _wav:
            g = npzparts.load(os.path.join(GOLDEN, "sample_full_pcm"))
            _wav["pcm"], _wav["sr"] = g["pcm_i16"].astype(np.float32) / 32768.0, int(g["sample_rate"])
        return oracle.frontend(cfg, _wav["pcm"], _wav["sr"], spectrum=False)["frames"]
    if inp["kind"] == "synth":
        p = synth_speech(inp["seconds"] * inp["sample_rate"], inp["sample_rate"], inp["seed"], inp["utt"])
        return oracle.frontend(cfg, p, inp["sample_rate"], spectrum=False)["frames"]
    if inp["kind"] == "adversarial":
        return adversarial_frames(inp["seed"], inp["B"], inp["F"])
    if inp["kind"] == "voiced_random":
        return voiced_random_frames(inp["seed"], inp["B"], inp["F"])
    if inp["kind"] == "dropped":
        return dropped_segment_frames()
    raise KeyError(inp["kind"])


def check_against_reference(case, an, level, step):
    """`an` = tables in the oracle's layout (oracle.Analysis, or the CUDA path's UtteranceResult-like)."""
    assert [list(x) for x in an.seg_ci] == case["seg_ci"]
    stored = [s for s in an.segments if s["stored"] >= 0]
    assert len(stored) == len([e for e in case["seg_ci"]]) - sum(1 for s in an.segments if s["stored"] < 0)
    if case["formants_sha"] is not None:
        assert an.formants.shape[0] == case["formant_rows"]
        assert sha(an.formants) == case["formants_sha"]
    else:
        assert an.formants.shape[0] == 0
    if case["syl_ci"] is not None:
        mine = [[[int(y["start"]), int(y["len"])] for y in an.syllables[s["first_syllable"]: s["first_syllable"] + s["n_syllables"]]]
                for s in stored]
        assert mine == case["syl_ci"]
    res = UtteranceResult({}, an.segments, an.formants, an.energy, an.syllables, an.features, getattr(an, "utterance", None),
                          getattr(an, "track_points", None))
    calls = api.segment_callbacks(level, step, DOC["labels"], res)
    assert len(calls) == len(case["events"])
    for mine, ref in zip(calls, case["events"]):
        assert mine[0] == ref[0] and mine[1] == ref[1]
        if level == 3:
            # b(e, label, s[e]): the ranked 18-field track arrays -- every number of every track (canonical JSON checksum)
            sys.path.insert(0, GOLDEN)
            from make_ref_js_golden import tracks_digest
            assert len(mine) == 3
            d = tracks_digest(mine[2])
            assert (d["tracks"], d["points"]) == (ref[2]["tracks"], ref[2]["points"]) and d["first"] == ref[2]["first"]
            assert d["sha"] == ref[2]["sha"]
            continue
        assert mine[2] == ref[2]                       # time stamps: numbers (4, 5) or toFixed(3) strings (10, 13)
        if level == 13:
            assert np.array_equal(np.array(mine[3], np.float64), np.array(ref[3], np.float64), equal_nan=True)
            assert all(len(r) == 53 for r in mine[3])
        elif level == 12:
            # 23 numbers per syllable: coefficients from numeric.uncmin, residual, point count -- doubles bit for bit
            assert [len(r) for r in mine[3]] == [len(r) for r in ref[3]] and all(len(r) == 23 for r in mine[3])
            a, b = np.array(mine[3], np.float64), np.array(ref[3], np.float64)
            assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), np.abs(a - b).max()
        elif level == 5:
            assert np.array_equal(np.array(mine[3], np.float64), np.array(ref[3], np.float64), equal_nan=True) and len(mine[3]) == 53
        elif level == 11:
            # cumulative 264-dim distributions (get_utterance_features @B107983), un-normalised histograms included
            assert np.array_equal(np.array(mine[3], np.float64), np.array(ref[3], np.float64), equal_nan=True) and len(mine[3]) == 264
        elif level == 4:
            a = np.stack(mine[3]).astype(np.float32)
            assert a.shape[0] == ref[3]["f32_rows"] and sha(a) == ref[3]["sha"]
        elif level == 10:
            assert len(mine[3]) == len(ref[3])
            for a, b in zip(mine[3], ref[3]):
                a = np.stack(a).astype(np.float32).reshape(-1, 9)
                assert a.shape[0] == b["f32_rows"] and sha(a) == b["sha"]


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_matches_reference_js(name):
    case = CASES[name]
    cfg = FaConfig.default(**case["kwargs"])
    fr = frames_for(case["input"], cfg)
    assert fr.shape == (case["frames"], case["bands"]) and sha(fr) == case["frames_sha"]   # same input as the reference saw
    an = oracle.analyze_frames(cfg, fr)
    check_against_reference(case, an, cfg.output_level, cfg.window_step_ms)


@pytest.mark.parametrize("name", list(CASES12))
def test_oracle_level12_matches_reference_js(name):
    """make_coeffs @B34527 / polyfit @B33793 with numeric.inv / uncmin / gradient (include/fa_curves.h) against what the
    reference's own code returned to its callback."""
    case = CASES12[name]
    cfg = FaConfig.default(**case["kwargs"])
    fr = frames_for(case["input"], cfg)
    assert fr.shape == (case["frames"], case["bands"]) and sha(fr) == case["frames_sha"]
    an = oracle.analyze_frames(cfg, fr)
    check_against_reference(case, an, 12, cfg.window_step_ms)


@pytest.mark.parametrize("name", list(CASES3))
def test_oracle_level3_matches_reference_js(name):
    """Level 3: what the reference handed to its callback -- get_ranked_formants @B35670 -- rebuilt from fa_track headers and
    fa_track_point rows by api.track_arrays."""
    case = CASES3[name]
    cfg = FaConfig.default(**case["kwargs"])
    fr = frames_for(case["input"], cfg)
    assert fr.shape == (case["frames"], case["bands"]) and sha(fr) == case["frames_sha"]
    an = oracle.analyze_frames(cfg, fr)
    check_against_reference(case, an, 3, cfg.window_step_ms)


def test_fixture_covers_the_quirks():
    """The vectors exercise: every callback level, dropped segments (seg_ci longer than the stores), multi-syllable
    segments, NaN features, the fixed noise gate."""
    levels = {FaConfig.default(**c["kwargs"]).output_level for c in DOC["cases"] if c["events"]}
    assert levels >= {4, 5, 10, 11, 13}
    assert any(len(c["seg_ci"]) > len(c["events"]) and c["kwargs"]["output_level"] in (4, 5, 13) for c in DOC["cases"])
    assert any(c["syl_ci"] and any(len(s) > 1 for s in c["syl_ci"]) for c in DOC["cases"])
    assert any(not c["kwargs"].get("auto_noise_gate", 1) and c["events"] for c in DOC["cases"])
    assert sum(len(c["seg_ci"]) for c in DOC["cases"]) > 150
    l11 = [c for c in DOC["cases"] if c["kwargs"]["output_level"] == 11 and c["events"]]
    assert any(max(np.sum(e[3]) for e in c["events"]) > 15.5 for c in l11)              # a poisoned (raw-count) histogram
    assert any(len(c["seg_ci"]) > len(c["events"]) for c in l11)                        # level 11 after a dropped segment


@pytest.mark.skipif(not run_reference.available(), reason="reference not mounted (GPU box): the committed vectors stand in")
def test_live_reference_run_reproduces_the_fixture():
    """Re-executes the reference's modules here on two cases and checks the committed vectors are what they produce."""
    sys.path.insert(0, GOLDEN)
    import make_ref_js_golden as gen
    R = run_reference.ReferenceModules()
    srcs = run_reference.module_sources()
    import hashlib
    for m, (off, src) in srcs.items():
        assert DOC["executed"][f"inner module {m}"]["sha256"] == hashlib.sha256(src.encode()).hexdigest()
    for name in ("synth_sr16000_seed1_u0_l13", "dropped_segment_l5", "voiced_random_seed7_B128_l5"):
        case = CASES[name]
        cfg = FaConfig.default(**case["kwargs"])
        fr = frames_for(case["input"], cfg)
        ref = R.analyze(fr, cfg.output_level, cfg.window_step_ms, bands=cfg.bands, plot_len=cfg.plot_len,
                        pause_ms=cfg.pause_length_ms, minlen_ms=cfg.min_seg_length_ms, auto_gate=bool(cfg.auto_noise_gate),
                        max_db=cfg.voiced_max_db, min_db=cfg.voiced_min_db, test_play=False, labels=DOC["labels"])
        assert ref["seg_ci"] == case["seg_ci"]
        got = json.loads(json.dumps([gen.encode_event(cfg.output_level, e) for e in ref["events"]]))
        want = case["events"]
        assert json.dumps(got) == json.dumps(want)


# ---------------------------------------------------------------------------- the interpreter itself
JS_SEMANTICS = {
    "1+2*3": 7.0, "(2**10)": 1024.0, "parseInt(.7*128)": 89.0, "[1,2,3].reduce(((e,t)=>e+t),0)/3": 2.0,
    "(function(){let e=[];e[0]=[1,2];e[1]=3;return e.length})()": 2.0,
    "(1.0005).toFixed(3)": "1.000", "(0.0625).toFixed(3)": "0.063", "(2.5).toFixed(0)": "3", "(12.3456).toFixed(3)": "12.346",
    "new Array(3).fill(0).concat([1],2).length": 5.0,
    "(function(){var n=0;for(let r in [5,6,7])n+=[5,6,7][r];return n})()": 18.0,
    "(()=>{let a=new Float32Array(2);a[0]=0.1;return a[0]})()": 0.10000000149011612,
    "(()=>{let a=new Float32Array(1);a[0]+=16777217;return a[0]})()": 16777216.0,
    "(()=>{let x=[1,2,3,4,5];let y=x.splice(1,2);return y.length*10+x.length})()": 23.0,
    "(()=>{let x=[1,3];x.splice(1,0,2);return x.join('')})()": "123",
    "typeof undefined": "undefined", "void 0===undefined": True, "!0": True, "0==!1": True, "-1/0": float("-inf"),
    "(()=>{let u=-1;return -1==u||0==u})()": True,
    "(()=>{function f(a,b=3){return a+b}return f(1)+f(1,1)})()": 6.0,
    "(()=>{try{let x;x[0]}catch(e){return 7}})()": 7.0,
    "(function e(n){return n<2?1:n*e(n-1)})(5)": 120.0,
    "(()=>{let i=0,j=0;for(;i<10;)i++,j+=2;return j})()": 20.0,
    "(()=>{let t=5;return t>7?1:t>6?2:t>4?3:4})()": 3.0,
    "(()=>{let a=[3,1,2];let n=a.length,m=-1/0;for(;n--;)a[n]>m&&(m=a[n]);return m})()": 3.0,
    "1+'a'": "1a", "''+1.5": "1.5", "(()=>{let e=0;return e+=2,e*=3,e})()": 6.0,
    "(()=>{let o={a:1,b:{c:2}};o.b.c++;return o.b.c+o.a})()": 4.0,
    "Math.log10(1000)": 3.0, "Math.pow(10,2)": 100.0, "Math.sqrt(16)": 4.0, "parseInt(-3.7)": -3.0, "parseInt(1e-7)": 1.0,
    "(()=>{let c=0;do{c++}while(c<3);return c})()": 3.0,
    "(()=>{switch(2){case 1:return 1;case 2:return 5;default:return 9}})()": 5.0,
    # hist[NaN]++ creates a named property that for-in visits (get_utterance_features relies on it, @B109452)
    "(()=>{let h=[1,2];h[parseInt(0/0)]++;let t=0;for(let n in h)t+=h[n];return t!=t})()": True,
    "(()=>{let h=[1,2];h[-1]++;return h.slice().length+h.length})()": 4.0,
    "(()=>{let a=[1,2,3];for(let n=0;n<a.length;n++)a[n]/=2;return a[2]})()": 1.5,
    "[5,1,10].sort().join()": "1,10,5", "[5,1,10].sort((a,b)=>a-b).join()": "1,5,10",
    "(()=>{let e=[[1,2],[3,4]];return e[1][0]/e[0][1]})()": 1.5,
    "1/3+''": "0.3333333333333333", "1e21+''": "1e+21", "1.5e-7+''": "1.5e-7", "100+''": "100",
    "(()=>{var r=function(e,t){let n=0;for(let r=0;r<e.length;r++)n+=e[r]*Math.pow(t,r);return n};return r([1,2,3],2)})()": 17.0,
}


@pytest.mark.parametrize("src", list(JS_SEMANTICS))
def test_minijs_language_semantics(src):
    got = Interp().eval_expression(src)
    want = JS_SEMANTICS[src]
    assert type(got) is type(want) and got == want, (src, got, want)


def test_minijs_promise_ordering_and_executor_throw():
    it = Interp()
    it.run("var log=[];new Promise((r,j)=>{log.push(1);r(5)}).then(v=>{log.push(v)}).catch(e=>{log.push(-1)});log.push(2);")
    assert to_str(it.globals.vars["log"]) == "1,2"          # then-callbacks are micro-tasks
    it.run_microtasks()
    assert to_str(it.globals.vars["log"]) == "1,2,5"
    # a TypeError inside the executor rejects the promise (what drops a segment in O(), quirk 15)
    it.run("var l2=[];new Promise((r,j)=>{let x;x.y;r(1)}).then(v=>{l2.push(v)}).catch(e=>{l2.push(-1)});l2.push(2);")
    it.run_microtasks()
    assert to_str(it.globals.vars["l2"]) == "2,-1"
    it.run("var l3=[];window.setTimeout(function(){l3.push(9)},10);l3.push(1);")
    it.run_timers()
    assert to_str(it.globals.vars["l3"]) == "1,9"


def test_minijs_rejects_unsupported_syntax_loudly():
    for bad in ("class A{}", "let [a,b]=[1,2]", "f(...x)", "`t${1}`", "async function f(){await 1}"):
        with pytest.raises(SyntaxError):
            Interp().run(bad)


# ---------------------------------------------------------------------------- the public API module (boundary, SURVEY 8(b))
API_DOC = json.load(open(os.path.join(GOLDEN, "ref_js_api.json")))
REF_FIELDS = ("plot_enable", "spec_type", "output_level", "plot_len", "f_min", "f_max", "N_fft_bins", "N_mel_bins", "window_width",
              "window_step", "pause_length", "min_seg_length", "auto_noise_gate", "voiced_max_dB", "voiced_min_dB", "pre_norm_gain",
              "high_f_emph")


@pytest.mark.parametrize("k", range(len(API_DOC["configure"])))
def test_configure_mirror_matches_the_reference_module(k):
    """api.configure against what the reference's own configure() (@B3292, executed by minijs) leaves in its settings."""
    case = API_DOC["configure"][k]
    api.reset_defaults()
    api.configure(case["cfg"])
    mine, ref = api._settings, case["settings"]
    partial = not all(f in case["cfg"] for f in ("spec_type", "f_min", "high_f_emph", "auto_noise_gate", "voiced_min_dB"))
    for f in REF_FIELDS:
        if partial and ref[f] is None and f in ("spec_type", "f_min", "high_f_emph", "auto_noise_gate", "voiced_min_dB"):
            # the reference stores `undefined` for a `null !== x` field that is missing from the object (and then fails in
            # reset_nodes); the mirror keeps the previous value -- the one documented deviation (INTEGRATION.md)
            assert mine[f] == api._defaults()[f]
            continue
        assert mine[f] == ref[f], (f, mine[f], ref[f])
    api.reset_defaults()


def test_launch_rejections_and_argument_order_match_the_reference_module():
    by = {l["name"]: l for l in API_DOC["launch"]}
    # single-flight rule and the rejection strings
    assert by["already_playing"]["value"] == "Error: Already playing" and by["already_playing"]["calls"] == []
    assert by["file_without_source"]["value"] == by["unknown_source"]["value"] == "Invalid audio source"
    assert by["reset_nodes_rejects"]["value"] == "Invalid reset_nodes config"
    api.reset_defaults()
    api._state["playing"] = True
    assert str(api.LaunchAudioNodes(1, b"x").exception()) == by["already_playing"]["value"]
    api._state["playing"] = False
    assert str(api.LaunchAudioNodes(1, None).exception()) == by["file_without_source"]["value"]
    assert str(api.LaunchAudioNodes(5, b"x").exception()) == by["unknown_source"]["value"]
    # reset_segmentor(level, bands, plot_len, step, pause, min_len, auto_gate, max_dB, min_dB, callback, test_play, labels):
    # the argument order the oracle harness, the C-ABI config and the shims rely on
    rs = [c for c in by["file_online"]["calls"] if c[0] == "reset_segmentor"][0][1]
    assert rs[:9] == [13, 128, 200, 15, 200, 50, True, 100, 10] and rs[10] is False and rs[11] == ["lab"]
    rn = [c for c in by["file_online"]["calls"] if c[0] == "reset_nodes"][0][1]
    assert rn == [1, 50, 4000, 256, 128, 25, 15, 1000, 0]          # spec_type, f_min, f_max, fft bins, mel bins, width, step, gain, emph
    assert [c[0] for c in by["file_offline"]["calls"]][-2:] == ["Garbage_Collect", "offline_play_the_file"]
    assert by["file_offline"]["calls"][-1][1] == ["buffer", 0.5, 2.0]
    assert by["file_offline"]["calls"][1][1][10] is True          # test_play defaults to true: callbacks suppressed (quirk 13)
    api.reset_defaults()


@pytest.mark.skipif(not run_reference.available(), reason="reference not mounted")
def test_live_reference_api_module_reproduces_the_fixture():
    sys.path.insert(0, GOLDEN)
    import make_ref_js_api_golden as gen
    for case in API_DOC["configure"]:
        assert run_reference.ReferenceAPI().configure(case["cfg"]) == case["settings"]
    A = run_reference.ReferenceAPI()
    A.configure(dict(gen.FULL, output_level=13, window_step=15))
    st, val = A.launch(1, "buffer", None, ["lab"], False, False)
    want = [l for l in API_DOC["launch"] if l["name"] == "file_online"][0]
    assert (st, val) == (want["status"], want["value"]) and [[c[0], c[1]] for c in A.calls] == want["calls"]
