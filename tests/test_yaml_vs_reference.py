"""Differential test of the host layer's hydro.yaml parser (SURVEY f2) against the REFERENCE's own parser.

src/hydro_yaml_parser.cpp + hydro_types.h are the one piece of the reference that builds from its own sources (SURVEY.md
8c).  oracle/Makefile compiles them where they lie into oracle/_ref/ref_yaml_dump (and the same dump driver over this
repo's parser into oracle/_ref/our_yaml_dump); both print every field of the YAMLHydroData that ReadHydroYAML returns, or
EXCEPTION.  The corpus: every *.hydro.yaml shipped with the reference plus synthetic files that walk the parser's branches
(scalar period and its synonyms, amplitude vs height, inline / block sweeps, booleans, quoting, comments, per-body and
system-wide TaperedDirect options, the convolution section, malformed numbers, missing sections).

Known deviation, asserted here: BLOCK-form period sweeps

    period:
      range: { start: 10.0, stop: 13.0, step: 1.0, inclusive: true }

are rejected by the reference snapshot ("waves.period: invalid or empty specification") -- its period-block exit test
(`indent <= period_block_indent`, hydro_yaml_parser.cpp:537-540) fires on the `period:` line itself, so the nested keys
of :441-524 are never reached, and its own demos/yaml/f3of/f3of_rao.hydro.yaml does not load.  This repo's parser
implements the documented format (the sweep feeds the ensemble's batch axis, SetupHydroSweepFromYAML); everything else
is identical.

What the reference's parser prints for the synthetic, block-form and fuzzed files is stored in
tests/golden/yaml_reference_dumps.json.gz (tests/golden/make_fixtures.py records it from a reference build), so those
comparisons run everywhere; only the comparison over the reference's own *.hydro.yaml files needs the reference source
tree and skips without it.  CPU only."""
import glob
import gzip
import json
import os
import random
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "ref_yaml_dump")
OUR_BIN = os.path.join(ROOT, "oracle", "_ref", "our_yaml_dump")
REF_TREE = "/root/reference"
GOLDEN = os.path.join(ROOT, "tests", "golden", "yaml_reference_dumps.json.gz")

BASE = """hydrodynamics:
  bodies:
    - name: body1
      h5_file: hydroData/sphere.h5
%(body)s
  waves:
%(waves)s
%(extra)s
"""
REG = "    type: regular\n    height: 1\n    period: 5"
CASES = {
    "scalar": dict(waves="    type: regular\n    height: 2.0\n    period: 8.0\n    direction: 10\n    phase: 0.5"),
    "synonyms_T": dict(waves="    type: regular\n    H: 1.5\n    T: 7.5"),
    "synonyms_Tp": dict(waves="    type: irregular\n    h: 2.5\n    Tp: 9.0\n    spectrum: jonswap\n    seed: 42"),
    "synonyms_p": dict(waves="    type: regular\n    a: 0.75\n    p: 6"),
    "amp_and_height": dict(waves="    type: regular\n    a: 0.75\n    height: 3.0\n    period: 6"),
    "amplitude_word": dict(waves="    type: regular\n    amplitude: 0.5\n    period: 6"),
    "inline_values": dict(waves="    type: regular\n    height: 1\n    period: { values: [6.0, 7.5, 9] }"),
    "inline_values_list": dict(waves="    type: regular\n    height: 1\n    period: [6.0, 7.5, 9]"),
    "inline_linspace": dict(waves="    type: regular\n    height: 1\n    period: { linspace: { start: 2.0, stop: 5.0, num: 4 } }"),
    "inline_range": dict(waves="    type: regular\n    height: 1\n    period: { range: { start: 2.0, stop: 5.0, step: 1.0 } }"),
    "no_wave": dict(waves="    type: no_wave"),
    "still": dict(waves="    type: still"),
    "quoted": dict(waves="    type: \"irregular\"\n    height: '2.0'\n    period: \"8.0\"   # trailing comment\n"
                         "    spectrum: 'pierson_moskowitz'"),
    "bools": dict(waves=REG, body="      include_excitation: no\n      include_radiation: Off\n"
                                  "      radiation_calculation: state_space"),
    "bools2": dict(waves=REG, body="      include_excitation: TRUE\n      include_radiation: 0"),
    "body_td": dict(waves=REG, body="      radiation_convolution_mode: TaperedDirect\n      td_smoothing: moving_average\n"
                                    "      td_window_length: 9\n      td_rms_threshold_factor: 0.05\n"
                                    "      td_taper_fraction_remaining: 0.4\n      td_export_plot_csv: true"),
    "global_td": dict(waves=REG, extra="  radiation_convolution_mode: TaperedDirect\n  td_smoothing: moving_average\n"
                                       "  td_window_length: 11\n  td_export_plot_csv: yes"),
    "conv_section": dict(waves=REG, extra="  convolution:\n    mode: TaperedDirect\n    smoothing:\n      type: moving_average\n"
                                          "      window_length: 9\n      order: 2\n    taper:\n      start_percent: 0.6\n"
                                          "      end_percent: 0.9\n      final_amplitude: 0.05\n      end_time: 20\n"
                                          "    diagnostics:\n      export_csv: on"),
    "conv_smoothing_inline": dict(waves=REG, extra="  convolution:\n    mode: Baseline\n    smoothing: sg"),
    "bad_numbers": dict(waves="    type: regular\n    height: abc\n    period: 5x\n    direction: \n    seed: notanint"),
    "zero_period": dict(waves="    type: regular\n    height: 1\n    period: 0"),
    "neg_period": dict(waves="    type: regular\n    height: 1\n    period: -3"),
    "no_period_regular": dict(waves="    type: regular\n    height: 1"),
    "two_bodies": dict(waves=REG, body="    - name: body2\n      h5_file: /abs/path/x.h5\n      include_excitation: false"),
    "tabs_and_spaces": dict(waves="    type:   regular   \n    height:\t1\n    period: 5"),
    "empty_waves": dict(waves="    # nothing"),
    "uppercase_keys": dict(waves="    Type: regular\n    Height: 2\n    Period: 4\n    Direction: 3\n    Phase: 1\n    Seed: 5\n"
                                 "    Spectrum: jonswap"),
    "linspace_bad": dict(waves="    type: regular\n    height: 1\n    period: { linspace: { start: 2.0, stop: 5.0, num: 1 } }"),
    "range_bad": dict(waves="    type: regular\n    height: 1\n    period: { range: { start: 5.0, stop: 2.0, step: 1.0 } }"),
    "values_empty": dict(waves="    type: regular\n    height: 1\n    period: { values: [] }"),
    "range_noninteger": dict(waves="    type: regular\n    height: 1\n    period: { range: { start: 1.0, stop: 2.05, step: 0.3 } }"),
}
RAW = {
    "no_hydro_key": "model:\n  x: 1\n",
    "empty": "",
    "nobodies": "hydrodynamics:\n  waves:\n    type: regular\n    height: 1\n    period: 3\n",
}
# block-form sweeps: the known deviation (see the module docstring) -> expected period_values of THIS parser
BLOCK = {
    "block_values": ("    type: regular\n    height: 1\n    period:\n      values: [6.0, 7.0]", "period_values 2: 6 7"),
    "block_linspace": ("    type: regular\n    height: 1\n    period:\n      linspace: { start: 2.0, stop: 5.0, num: 4 }",
                       "period_values 4: 2 3 4 5"),
    "block_range_excl": ("    type: regular\n    height: 1\n    period:\n      range: { start: 2.0, stop: 5.0, step: 1.0, "
                         "inclusive: false }", "period_values 3: 2 3 4"),
    "block_range_incl": ("    type: regular\n    height: 1\n    period:\n      #values: [6.0, 7.0, 8.0, 9.0]\n"
                         "      range: { start: 10.0, stop: 13.0, step: 1.0, inclusive: true }", "period_values 4: 10 11 12 13"),
}


@pytest.fixture(scope="module")
def our_dumper():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    return OUR_BIN


@pytest.fixture(scope="module")
def reference():
    """The reference parser's output over this module's corpus: {"synthetic": {name: stdout}, "block": {name: [stdout,
    stderr]}, "fuzz": stdout}, with the corpus directory written as <dir>."""
    with gzip.open(GOLDEN, "rt") as f:
        return json.load(f)


@pytest.fixture(scope="module")
def dumpers(our_dumper):
    if not os.path.exists(REF_BIN):
        pytest.skip("the reference tree is not present here: no reference parser to compare with")
    return REF_BIN, OUR_BIN


def _dump(binary, path):
    out = subprocess.run([binary, str(path)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return out.stdout, out.stderr


def dump_in(binary, paths, d):
    """stdout, stderr of `binary` over `paths`, with the corpus directory d written as <dir> (the parsers resolve h5_file
    against the canonical directory of the hydro.yaml, so "../x.h5" comes out under the parent of d: <dir>/..)."""
    out = subprocess.run([binary] + [str(p) for p in paths], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr

    def norm(s):
        for p, name in ((d, "<dir>"), (d.resolve(), "<dir>"), (d.resolve().parent, "<dir>/..")):
            s = s.replace(str(p), name)
        return s
    return norm(out.stdout), norm(out.stderr)


def synthetic_corpus(d):
    """CASES and RAW written into directory d, plus a file name that does not exist: {name: path}."""
    texts = {name: BASE % dict(body=c.get("body", ""), waves=c["waves"], extra=c.get("extra", ""))
             for name, c in CASES.items()}
    texts.update(RAW)
    files = {}
    for name, text in texts.items():
        files[name] = d / (name + ".hydro.yaml")
        files[name].write_text(text)
    files["missing"] = d / "missing.hydro.yaml"
    return files


def block_corpus(d):
    files = {}
    for name, (waves, _) in BLOCK.items():
        files[name] = d / (name + ".hydro.yaml")
        files[name].write_text(BASE % dict(body="", waves=waves, extra=""))
    return files


def fuzz_corpus(d):
    """600 seeded random hydro.yaml files (inline forms only: block-form sweeps are the known deviation)."""
    rnd = random.Random(11)
    files = []
    for n in range(600):
        files.append(d / ("g%04d.hydro.yaml" % n))
        files[-1].write_text(_fuzz_file(rnd))
    return files


def test_synthetic_corpus_parses_identically(our_dumper, reference, tmp_path):
    ref = reference["synthetic"]
    files = synthetic_corpus(tmp_path)
    assert sorted(files) == sorted(ref)
    for name, f in files.items():
        r, o = ref[name], dump_in(our_dumper, [f], tmp_path)[0]
        assert r == o, "%s:\n--- reference\n%s--- this repo\n%s" % (name, r, o)
    assert "EXCEPTION" in ref["missing"]
    n_exc = sum("EXCEPTION" in r for name, r in ref.items() if name != "missing")
    assert 8 <= n_exc < len(files) - 1 - 15      # the corpus exercises both the accepting and the throwing branches


def test_reference_yaml_files_parse_identically(dumpers):
    ref, our = dumpers
    if not os.path.isdir(REF_TREE):
        pytest.skip("the reference tree is not present here")
    files = sorted(glob.glob(os.path.join(REF_TREE, "**", "*.hydro.yaml"), recursive=True))
    assert len(files) >= 10
    deviating = []
    for f in files:
        r, o = _dump(ref, f)[0], _dump(our, f)[0]
        if r != o:
            deviating.append(os.path.basename(f))
            assert "EXCEPTION" in r and "period_values 4: 10 11 12 13" in o, f      # the block-form sweep, nothing else
    assert deviating in ([], ["f3of_rao.hydro.yaml"]), deviating


def test_block_form_sweeps_are_the_one_known_deviation(our_dumper, reference, tmp_path):
    files = block_corpus(tmp_path)
    assert sorted(files) == sorted(reference["block"])
    for name, f in files.items():
        r, rerr = reference["block"][name]
        o, _ = dump_in(our_dumper, [f], tmp_path)
        assert "EXCEPTION" in r and "invalid or empty specification" in rerr, name
        assert BLOCK[name][1] in o.splitlines(), (name, o)


def _fuzz_file(rnd):
    def num():
        return rnd.choice(["2.0", "0", "-1", "1e1", "3.25", "12", "0.5", "  7  ", "'3.5'", "\"4\"", "5 # c", "abc", ""])
    L = ["hydrodynamics:", "  bodies:"]
    for b in range(rnd.randint(1, 3)):
        L.append("    - name: body%d" % (b + 1))
        L.append("      h5_file: %s" % rnd.choice(["x.h5", "/a/b.h5", "../d/e.h5", "'q.h5'"]))
        for k, vs in [("include_excitation", ["true", "false", "no", "On", "0", "1", "Yes", "maybe"]),
                      ("include_radiation", ["true", "false", "off"]), ("radiation_calculation", ["convolution", "state_space"]),
                      ("radiation_convolution_mode", ["TaperedDirect", "Baseline"]), ("td_smoothing", ["sg", "moving_average"]),
                      ("td_window_length", ["7", "abc", "3"]), ("td_rms_threshold_factor", ["0.1", "x"]),
                      ("td_taper_fraction_remaining", ["0.3"]), ("td_export_plot_csv", ["true", "no"])]:
            if rnd.random() < 0.3:
                L.append("      %s: %s" % (k, rnd.choice(vs)))
    L.append("  waves:")
    L.append("    type: %s" % rnd.choice(["regular", "irregular", "no_wave", "still", "Regular", "IRREGULAR"]))
    W = []
    if rnd.random() < 0.8:
        W.append("%s: %s" % (rnd.choice(["height", "h", "H"]), num()))
    if rnd.random() < 0.4:
        W.append("%s: %s" % (rnd.choice(["a", "amplitude", "A"]), num()))
    r, pk = rnd.random(), rnd.choice(["period", "T", "Tp", "p", "Period"])
    if r < 0.5:
        W.append("%s: %s" % (pk, num()))
    elif r < 0.65:
        W.append("%s: { values: [%s] }" % (pk, ", ".join(rnd.choice(["4", "5.5", "6", "x"]) for _ in range(rnd.randint(0, 4)))))
    elif r < 0.75:
        W.append("%s: { linspace: { start: 1, stop: %s, num: %s } }" % (pk, rnd.choice(["2", "0"]), rnd.choice(["3", "1", "x"])))
    elif r < 0.85:
        W.append("%s: { range: { start: 1, stop: %s, step: %s, inclusive: %s } }"
                 % (pk, rnd.choice(["2", "0", "2.05"]), rnd.choice(["0.5", "0", "0.3"]), rnd.choice(["true", "false"])))
    for k in ["direction", "phase", "spectrum", "seed"]:
        if rnd.random() < 0.5:
            W.append("%s: %s" % (k, rnd.choice(["jonswap", "pierson_moskowitz"]) if k == "spectrum" else num()))
    rnd.shuffle(W)
    L += ["    " + w for w in W]
    if rnd.random() < 0.3:
        L += ["  convolution:", "    mode: %s" % rnd.choice(["TaperedDirect", "Baseline"])]
        if rnd.random() < 0.6:
            L += ["    smoothing:", "      type: %s" % rnd.choice(["sg", "moving_average", "savitzky_golay"]),
                  "      window_length: %s" % rnd.choice(["5", "9", "x"])]
        if rnd.random() < 0.6:
            L += ["    taper:", "      start_percent: %s" % rnd.choice(["0.5", "x"]), "      end_percent: 0.9",
                  "      final_amplitude: 0.1", "      end_time: %s" % rnd.choice(["10", "-1"])]
        if rnd.random() < 0.6:
            L += ["    diagnostics:", "      export_csv: %s" % rnd.choice(["true", "no"])]
    if rnd.random() < 0.3:
        for k, vs in [("radiation_convolution_mode", ["TaperedDirect", "Baseline"]), ("td_smoothing", ["sg", "moving_average"]),
                      ("td_window_length", ["7", "x"]), ("td_export_plot_csv", ["true", "0"])]:
            if rnd.random() < 0.5:
                L.append("  %s: %s" % (k, rnd.choice(vs)))
    if rnd.random() < 0.15:
        L.insert(rnd.randint(1, len(L)), "    # comment")
    return "\n".join(L) + "\n"


def test_fuzzed_corpus_parses_identically(our_dumper, reference, tmp_path):
    """The fuzzed corpus: the two parsers print the same structure, or both throw, for every one of the files."""
    r = reference["fuzz"]
    o = dump_in(our_dumper, fuzz_corpus(tmp_path), tmp_path)[0]
    assert r == o
    n_exc = r.count("EXCEPTION")
    assert 100 < n_exc < 500, n_exc          # both outcomes are well represented
