"""The NMCH / exploration command line tools (C++ over the method API over the C ABI)."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NMCH = os.path.join(ROOT, "bin", "NMCH")
EXPL = os.path.join(ROOT, "bin", "exploration")


@pytest.fixture(scope="module", autouse=True)
def _built():
    from nmch_b200 import _build
    _build.build_cli(only_if_missing=True)
    assert os.path.exists(NMCH) and os.path.exists(EXPL)


def run(exe, *args):
    return subprocess.run([exe, *map(str, args)], capture_output=True, text=True, timeout=900)


def test_help_and_unknown_method_exit_codes():
    r = run(NMCH, "--help")
    assert r.returncode == 0 and "--method <string>  Method to use: fe or em (default: fe)" in r.stdout   # nmch.cu:94-111
    r = run(NMCH, "--method", "heun")
    assert r.returncode == 1 and r.stdout.strip() == "Unknown method: heun"                                # nmch.cu:135-137
    assert run(EXPL, "--help").returncode == 0


def test_error_convention_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = run(NMCH, "--NB", 8)
    assert r.returncode == 1
    assert re.search(r"There is an error in file .* at line \d+", r.stdout)     # utils.cu:30-35
    assert "no CPU fallback" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("method,title", [("fe", "FORWARD-EULER"), ("em", "EXACT-METHOD")])
def test_nmch_report_matches_reference_format(method, title):
    r = run(NMCH, "--method", method, "--NB", 64, "--N", 200, "--json")
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    want = ["Base parameters:", "NTPB    = 512", "NB      = 64", "T       = 1.000000", "S_0,K   = 1.000000",
            "v_0     = 0.100000", "r       = 0.000000", "k       = 0.500000", "theta   = 0.100000",
            "sigma   = 0.300000", "N       = 200", "dt      = 0.005000", f"METHOD: {title}"]
    assert lines[:13] == want
    assert lines[13].startswith("The estimated price E[X] is equal to ")
    assert lines[14].startswith("The estimated E[X^2] is equal to ")
    assert lines[15] == "The true price 0.119235"                                   # Black-Scholes line, NMCH_FE.cu:336-338
    assert lines[16].startswith("error associated to a confidence interval of 95% = ")
    assert lines[17].startswith("Execution time ") and lines[17].endswith(" ms")
    assert lines[18].startswith("Initialization time ")
    j = json.loads(lines[19])
    from nmch_b200 import engine as E
    with E.Engine(NTPB=512, NB=64, N=200, method=E.METHOD_FE if method == "fe" else E.METHOD_EM) as e:
        e.init(1234)
        m = e.compute()
    assert j["sum_payoff"] == m.sum_payoff and j["sum_payoff_sq"] == m.sum_payoff_sq
    assert abs(float(lines[13].split()[-1]) - m.mean) < 1e-6


@pytest.mark.gpu
def test_nmch_xorwow_tag_matches_reference_binary():
    from ref_build import harness_rows
    r = run(NMCH, "--rng", "xorwow", "--NB", 128, "--N", 300, "--json")
    j = json.loads(r.stdout.splitlines()[-1])
    ref = harness_rows(method="fe", rng="xorwow", NB=128, N=300)[0]
    assert abs(j["E"] - ref["E"]) / ref["E"] < 1e-5
    assert abs(j["err"] - ref["err"]) / ref["err"] < 1e-4          # the reference's own CI formula, same inputs


@pytest.mark.gpu
def test_nmch_opt_in_stream_modes():
    """--rng xorwow-fast: the reference's draws, native arithmetic (same price as the reference binary to 1e-5);
    --rng philox-dense: own mapping (statistical agreement); both are FE-only and say so for --method em."""
    from oracle import oracle as o
    j = json.loads(run(NMCH, "--rng", "xorwow-fast", "--NB", 128, "--N", 300, "--json").stdout.splitlines()[-1])
    if os.path.exists(o.REF_HARNESS_PATH):
        ref = json.loads(run(o.REF_HARNESS_PATH, "--method", "fe", "--rng", "xorwow", "--NB", 128, "--N", 300).stdout.splitlines()[0])
        assert abs(j["E"] - ref["E"]) / ref["E"] < 1e-5
    c = json.loads(run(NMCH, "--rng", "xorwow", "--NB", 128, "--N", 300, "--json").stdout.splitlines()[-1])
    assert abs(j["E"] - c["E"]) / c["E"] < 1e-5 and j["rng"] == "xorwow-fast"
    d = json.loads(run(NMCH, "--rng", "philox-dense", "--NB", 2048, "--N", 300, "--json").stdout.splitlines()[-1])
    p = json.loads(run(NMCH, "--rng", "philox", "--NB", 2048, "--N", 300, "--json").stdout.splitlines()[-1])
    assert abs(d["E"] - p["E"]) < 3 * np.hypot(d["std_error"], p["std_error"])
    for mode in ("xorwow-fast", "philox-dense"):                   # FE-only stream modes
        r = run(NMCH, "--method", "em", "--rng", mode, "--NB", 8, "--N", 10)
        assert r.returncode == 1 and "forward-Euler stream mode" in r.stdout


@pytest.mark.gpu
def test_exploration_default_run_is_the_reference_sweep():
    from oracle import oracle as o
    r = run(EXPL, "--N", 40)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    assert lines[0] == "method, k, theta, sigma, execution_time, err"              # exploration.cu:69
    fe = [l.split(", ") for l in lines[1:] if l.startswith("fe")]
    em = [l.split(", ") for l in lines[1:] if l.startswith("em")]
    k, th, sg = o.exploration_grid(5, apply_filter=True)
    assert len(fe) == len(em) == len(k) == 200
    np.testing.assert_allclose([float(x[1]) for x in fe], k, atol=1e-6)
    np.testing.assert_allclose([float(x[3]) for x in fe], sg, atol=1e-6)
    # same err column as the reference build for the first points (XORWOW tag, continued streams, N = 40)
    if os.path.exists(o.REF_HARNESS_PATH):
        import tempfile
        pts = os.path.join(tempfile.mkdtemp(), "sweep_pts.txt")
        with open(pts, "w") as f:
            f.write("0.5 0.1 0.3\n")                                                 # the warm-up compute
            for i in range(8):
                f.write(f"{k[i]:.9g} {th[i]:.9g} {sg[i]:.9g}\n")
        ref = [json.loads(l) for l in run(o.REF_HARNESS_PATH, "--method", "fe", "--rng", "xorwow", "--NTPB", 512, "--NB", 10,
                                          "--N", 40, "--points", pts).stdout.splitlines()][1:]
        for i in range(8):
            assert abs(float(fe[i][5]) - ref[i]["err"]) <= 2e-6 + 1e-4 * ref[i]["err"], (i, fe[i], ref[i]["err"])


@pytest.mark.gpu
def test_exploration_bias_column_and_linspace_grid():
    r = run(EXPL, "--points", 3, "--log2-paths", 16, "--N", 400, "--rng", "philox", "--method", "fe", "--bias")
    assert r.returncode == 0, r.stderr
    rows = [l.split(", ") for l in r.stdout.splitlines()[1:]]
    assert r.stdout.splitlines()[0].endswith(", bias")
    assert 20 <= len(rows) <= 27
    # the CSV is what the reference's heatmap.py consumes: columns method/k/theta/sigma/bias after stripping blanks
    import io
    import pandas as pd
    df = pd.read_csv(io.StringIO(r.stdout))
    df.columns = df.columns.str.strip()
    assert {"method", "k", "theta", "sigma", "bias"} <= set(df.columns) and len(df) == len(rows)
    assert pd.to_numeric(df["bias"], errors="coerce").notna().all()
    worst = max(rows, key=lambda x: abs(float(x[6])))
    assert abs(float(worst[6])) < 0.03, worst                  # Euler bias (sigma = 1 corners) + MC noise stay small


# ---------------------------------------------------------------------------------------------------------------------
# Text-level drop-in check against the reference's OWN command line tools: oracle/_ref/nmch_ref_cli and
# oracle/_ref/nmch_ref_exploration are src/NMCH/test/nmch.cu and exploration.cu compiled unmodified (oracle/Makefile).
# Same command line in, same text out -- up to the last printed digit of the estimates (float atomics on their side) and
# the two timing lines.
# ---------------------------------------------------------------------------------------------------------------------
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "nmch_ref_cli")
REF_EXPL = os.path.join(ROOT, "oracle", "_ref", "nmch_ref_exploration")


def _same_text_close_number(ours, ref, abs_tol, rel_tol):
    a, b = ours.rsplit(" ", 1), ref.rsplit(" ", 1)
    assert a[0] == b[0], (ours, ref)
    x, y = float(a[1]), float(b[1])
    assert abs(x - y) <= abs_tol + rel_tol * abs(y), (ours, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("args,extra", [
    (("--method", "fe", "--NB", 64, "--N", 200), ()),                          # Philox tag -> our default fast mode
    (("--method", "fe", "--NB", 64, "--N", 200), ("--rng", "philox-compat")),  # ... and the draw-compatible checker
    (("--method", "fe", "--NTPB", 256, "--NB", 128, "--N", 365, "--T", 0.5, "--S_0", 2.0, "--v_0", 0.04, "--r", 0.03, "--k", 1.5,
      "--rho", 0.3, "--theta", 0.09, "--sigma", 0.5, "--seed", 77), ()),
    (("--method", "em", "--NB", 64, "--N", 200), ("--rng", "philox-compat")),  # the reference's EM draws (its bias included)
])
def test_nmch_prints_what_the_reference_cli_prints(args, extra):
    if not os.path.exists(REF_CLI):
        pytest.skip("oracle/_ref/nmch_ref_cli not shipped")
    ref = run(REF_CLI, *args)
    ours = run(NMCH, *args, *extra)
    assert ref.returncode == 0 and ours.returncode == 0, (ref.stderr, ours.stderr)
    r, o_ = ref.stdout.splitlines(), ours.stdout.splitlines()
    assert len(r) == len(o_) == 19
    assert o_[:13] == r[:13]                                   # parameter block and METHOD line, byte for byte
    _same_text_close_number(o_[13], r[13], 2e-6, 1e-5)         # E[X]
    _same_text_close_number(o_[14], r[14], 2e-6, 1e-5)         # E[X^2]
    assert o_[15] == r[15]                                     # "The true price ..." (their Black-Scholes line)
    _same_text_close_number(o_[16], r[16], 2e-6, 1e-4)         # 95 % error
    for i in (17, 18):                                         # timings: same words, own numbers
        assert o_[i].rsplit(" ", 2)[0] == r[i].rsplit(" ", 2)[0] and o_[i].endswith(" ms")


@pytest.mark.gpu
def test_nmch_help_and_errors_read_like_the_reference():
    if not os.path.exists(REF_CLI):
        pytest.skip("oracle/_ref/nmch_ref_cli not shipped")
    r, o_ = run(REF_CLI, "--help"), run(NMCH, "--help")
    assert r.returncode == o_.returncode == 0
    rl, ol = r.stdout.splitlines(), o_.stdout.splitlines()
    assert ol[1:len(rl)] == rl[1:]                             # every reference line, in order (ours adds flags after them)
    assert rl[0].startswith("Usage: ") and ol[0].startswith("Usage: ")
    r, o_ = run(REF_CLI, "--method", "heun"), run(NMCH, "--method", "heun")
    assert (r.returncode, r.stdout) == (o_.returncode, o_.stdout)


@pytest.mark.gpu
def test_exploration_prints_what_the_reference_exploration_prints():
    """The reference's tool takes no arguments (512 x 10 paths, N = 1000, seed 1234, XORWOW tag, 200 FE + 200 EM points on
    continued streams).  Ours, run without arguments, must print the same CSV: same header, same rows in the same order with
    byte-identical method / k / theta / sigma fields, the err column equal to the printed precision (FE: all 200 rows; EM:
    the draw-compatible stream reproduces the reference's accept/reject decisions, so its rows match too)."""
    if not os.path.exists(REF_EXPL):
        pytest.skip("oracle/_ref/nmch_ref_exploration not shipped")
    ref, ours = run(REF_EXPL), run(EXPL)
    assert ref.returncode == 0 and ours.returncode == 0, (ref.stderr, ours.stderr)
    r, o_ = ref.stdout.splitlines(), ours.stdout.splitlines()
    assert o_[0] == r[0] and len(o_) == len(r) == 401
    worst = {"fe": 0.0, "em": 0.0}
    for a, b in zip(o_[1:], r[1:]):
        fa, fb = a.split(", "), b.split(", ")
        assert fa[:4] == fb[:4], (a, b)
        assert len(fa) == len(fb) == 6
        d = abs(float(fa[5]) - float(fb[5])) / float(fb[5])
        worst[fa[0]] = max(worst[fa[0]], d)
    # err ~ 5e-3 printed with 6 decimals: one unit of the last digit is 2e-4 relative
    assert worst["fe"] < 4e-4, worst
    assert worst["em"] < 4e-4, worst
