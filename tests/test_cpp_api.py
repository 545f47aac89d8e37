"""The C++ method API is source-compatible with reference-style user code (reference README.md:60-93) and links
with plain g++ (no nvcc, no curand headers on the user side)."""
import os
import subprocess
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

USER_CODE = textwrap.dedent(r"""
    #include "NMCH/methods/NMCH_FE.hpp"
    #include "NMCH/methods/NMCH_EM.hpp"
    #include <cstring>
    using namespace nmch::methods;

    template <typename M> static int drive(int NTPB, int NB, int N)
    {
        M nmch(NTPB, NB, 1.0f, 1.0f, 0.1f, 0.0f, 0.5f, -0.7f, 0.1f, 0.3f, N);
        nmch.init(1234ULL);
        nmch.compute();
        nmch.set_k(1.0f); nmch.set_theta(0.2f); nmch.set_sigma(0.4f);
        nmch.compute();
        nmch.print_stats();
        float e = nmch.get_strike_price(), e2 = nmch.get_price_squared(), t = nmch.get_execution_time(), err = nmch.get_err();
        nmch.finalize();
        return (e > 0 && e2 > 0 && t >= 0 && err > 0) ? 0 : 3;
    }

    int main(int argc, char **argv)
    {
        if (argc > 1 && !strcmp(argv[1], "types")) return 0;      // compile/link check only
        int rc = 0;
        rc |= drive<NMCH_FE_K1_MM<curandStateXORWOW_t>>(128, 8, 50);
        rc |= drive<NMCH_FE_K2_MM<curandStatePhilox4_32_10_t>>(128, 8, 50);
        rc |= drive<NMCH_FE_K3_MM<curandStateMRG32k3a_t>>(128, 8, 50);
        rc |= drive<NMCH_FE_K2_PHILOX_MM>(128, 8, 50);
        rc |= drive<NMCH_FE_K1_PgM<curandStateXORWOW_t>>(128, 8, 50);
        rc |= drive<NMCH_FE_K1_PiM<curandStateXORWOW_t>>(128, 8, 50);
        rc |= drive<NMCH_EM_K1_MM<curandStateXORWOW_t>>(128, 8, 50);
        rc |= drive<NMCH_EM_K2_MM<curandStatePhilox4_32_10_t>>(128, 8, 50);
        rc |= drive<NMCH_EM_K3_MM<curandStateXORWOW_t>>(128, 8, 50);
        return rc;
    }
""")


@pytest.fixture(scope="module")
def user_exe(tmp_path_factory):
    from nmch_b200 import _build
    _build.build(only_if_missing=True)
    d = tmp_path_factory.mktemp("user")
    src = d / "user.cpp"
    src.write_text(USER_CODE)
    exe = d / "user"
    api = [os.path.join(ROOT, "src", "NMCH", "methods", f) for f in ("NMCH.cpp", "NMCH_FE.cpp", "NMCH_EM.cpp")]
    api.append(os.path.join(ROOT, "src", "NMCH", "utils", "utils.cpp"))
    pkg = os.path.join(ROOT, "nmch_b200")
    subprocess.run(["/usr/bin/g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), *api, "-o",
                    str(exe), "-L", pkg, "-lnmch_b200", f"-Wl,-rpath,{pkg}"], check=True)
    return str(exe)


def test_reference_style_user_code_compiles_and_links(user_exe):
    assert subprocess.run([user_exe, "types"]).returncode == 0


@pytest.mark.gpu
def test_all_reference_class_names_run(user_exe):
    r = subprocess.run([user_exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
    assert r.stdout.count("METHOD: FORWARD-EULER") == 6 and r.stdout.count("METHOD: EXACT-METHOD") == 3


def test_heston_pricer_in_utils_matches_oracle(tmp_path):
    from oracle import oracle as o
    src = tmp_path / "h.cpp"
    src.write_text('#include "NMCH/utils/utils.hpp"\n#include <cstdio>\nint main(){printf("%.12f %.12f %.9f\\n",'
                   'nmch::utils::heston_call(1,1,0.1,0,0.5,0.1,0.3,-0.7,1), nmch::utils::heston_call(1,1,0.1,0,2.08,0.108,1.0,-0.7,1),'
                   'nmch::utils::NP(0.15));}')
    exe = tmp_path / "h"
    pkg = os.path.join(ROOT, "nmch_b200")
    subprocess.run(["/usr/bin/g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src),
                    os.path.join(ROOT, "src", "NMCH", "utils", "utils.cpp"), "-o", str(exe), "-L", pkg, "-lnmch_b200",
                    f"-Wl,-rpath,{pkg}"], check=True)
    a, b, c = map(float, subprocess.run([str(exe)], capture_output=True, text=True).stdout.split())
    assert abs(a - 0.1197325094) < 2e-9 and abs(b - 0.1104934558) < 2e-9
    assert abs(c - o.lib().orc_NP(0.15)) < 1e-9          # printed with 9 decimals


# ---------------------------------------------------------------------------------------------------------------------
# Every class name of the reference (NMCH_FE.hpp:21-189, NMCH_EM.hpp:19-128), through OUR C++ API, against the SAME class of
# the reference's CUDA build (oracle/_ref/nmch_ref_harness) on the same seed and two consecutive compute() calls.
# ---------------------------------------------------------------------------------------------------------------------
MATRIX_CODE = textwrap.dedent(r"""
    #include "NMCH/methods/NMCH_FE.hpp"
    #include "NMCH/methods/NMCH_EM.hpp"
    #include <cstdio>
    #include <cstdlib>
    #include <cstring>
    using namespace nmch::methods;

    template <typename M> static int drive(bool legacy, int NTPB, int NB, int N)
    {
        M nmch(NTPB, NB, 1.0f, 1.0f, 0.1f, 0.0f, 0.5f, -0.7f, 0.1f, 0.3f, N);
        nmch.set_legacy_k1_moment(legacy);
        nmch.init(1234ULL);
        for (int call = 0; call < 2; ++call) {
            nmch.compute();
            printf("{\"E\": %.9g, \"E2\": %.9g}\n", nmch.get_strike_price(), nmch.get_price_squared());
        }
        nmch.finalize();
        return 0;
    }

    #define TAGS(NAME, LEGACY)                                                                                  \
        if (!strcmp(argv[1], #NAME) && !strcmp(argv[2], "xorwow")) return drive<NAME<curandStateXORWOW_t>>(LEGACY, NTPB, NB, N);        \
        if (!strcmp(argv[1], #NAME) && !strcmp(argv[2], "philox")) return drive<NAME<curandStatePhilox4_32_10_t>>(LEGACY, NTPB, NB, N); \
        if (!strcmp(argv[1], #NAME) && !strcmp(argv[2], "mrg")) return drive<NAME<curandStateMRG32k3a_t>>(LEGACY, NTPB, NB, N);

    int main(int argc, char **argv)
    {
        if (argc < 6) return 2;
        const int NTPB = atoi(argv[3]), NB = atoi(argv[4]), N = atoi(argv[5]);
        TAGS(NMCH_FE_K1_MM, true)
        TAGS(NMCH_FE_K1_PgM, true)
        TAGS(NMCH_FE_K1_PiM, true)
        TAGS(NMCH_FE_K2_MM, false)
        TAGS(NMCH_FE_K3_MM, false)
        TAGS(NMCH_EM_K1_MM, true)
        TAGS(NMCH_EM_K2_MM, false)
        TAGS(NMCH_EM_K3_MM, false)
        if (!strcmp(argv[1], "NMCH_FE_K2_PHILOX_MM")) return drive<NMCH_FE_K2_PHILOX_MM>(false, NTPB, NB, N);
        return 2;
    }
""")


@pytest.fixture(scope="module")
def matrix_exe(tmp_path_factory):
    from nmch_b200 import _build
    _build.build(only_if_missing=True)
    d = tmp_path_factory.mktemp("matrix")
    src = d / "matrix.cpp"
    src.write_text(MATRIX_CODE)
    exe = d / "matrix"
    api = [os.path.join(ROOT, "src", "NMCH", "methods", f) for f in ("NMCH.cpp", "NMCH_FE.cpp", "NMCH_EM.cpp")]
    api.append(os.path.join(ROOT, "src", "NMCH", "utils", "utils.cpp"))
    pkg = os.path.join(ROOT, "nmch_b200")
    subprocess.run(["/usr/bin/g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), *api, "-o",
                    str(exe), "-L", pkg, "-lnmch_b200", f"-Wl,-rpath,{pkg}"], check=True)
    return str(exe)


def test_class_matrix_user_code_compiles(matrix_exe):
    assert subprocess.run([matrix_exe]).returncode == 2           # usage: no class named


_MATRIX = [("NMCH_FE_K1_MM", "fe", "k1", ("xorwow", "philox", "mrg")), ("NMCH_FE_K1_PgM", "fe", "k1pgm", ("xorwow", "philox")),
           ("NMCH_FE_K1_PiM", "fe", "k1pim", ("xorwow", "philox")), ("NMCH_FE_K2_MM", "fe", "k2", ("xorwow", "philox", "mrg")),
           ("NMCH_FE_K3_MM", "fe", "k3", ("xorwow", "philox", "mrg")), ("NMCH_FE_K2_PHILOX_MM", "fe", "k2philox", ("philox",)),
           ("NMCH_EM_K1_MM", "em", "k1", ("xorwow", "mrg")), ("NMCH_EM_K2_MM", "em", "k2", ("xorwow", "mrg")),
           ("NMCH_EM_K3_MM", "em", "k3", ("xorwow", "mrg"))]


@pytest.mark.gpu
@pytest.mark.parametrize("name,method,kernel,tags", _MATRIX, ids=[m[0] for m in _MATRIX])
def test_every_class_name_matches_the_same_class_of_the_reference_build(matrix_exe, name, method, kernel, tags):
    """FE: every tag (the Philox tag runs our default FAST mode on the reference's Philox words).  EM: the XORWOW and MRG tags
    are draw-compatible; the Philox tag of EM is our native exact sampler, a different (unbiased) stream by design, and is
    compared statistically elsewhere (tests/test_gpu_em.py).  K1-family classes with set_legacy_k1_moment(true): their
    price_squared is the reference's E[X^2]/n^2 (NMCH_FE.cu:56-58)."""
    import json
    from ref_build import harness_rows
    NTPB, NB, N = (256, 64, 120) if method == "fe" else (128, 32, 60)      # K1 needs a power-of-two block (NMCH_FE.cu:62-72)
    for tag in tags:
        want = harness_rows(timeout=600, method=method, rng=tag, kernel=kernel, NTPB=NTPB, NB=NB, N=N, repeat=2)
        ours = subprocess.run([matrix_exe, name, tag, str(NTPB), str(NB), str(N)], capture_output=True, text=True, timeout=600)
        assert ours.returncode == 0, ours.stdout[-400:] + ours.stderr[-400:]
        got = [json.loads(l) for l in ours.stdout.splitlines() if l.startswith("{")]
        assert len(got) == len(want) == 2
        for g, w in zip(got, want):
            assert abs(g["E"] - w["E"]) <= 2e-5 * abs(w["E"]), (name, tag, g, w)          # 16 k paths: float atomics + %.9g
            assert abs(g["E2"] - w["E2"]) <= 3e-5 * abs(w["E2"]), (name, tag, g, w)
