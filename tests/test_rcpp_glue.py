"""The literal drop-in: the product's src/bayesnet_mcmc.cpp + src/Makevars (bayesnetworks_b200/
csrc/rcpp_glue) built the way R CMD INSTALL would build them -- compile flags and link line taken
from the Makevars file -- against the stand-in Rcpp.h (R is not installed), then RUN through a
driver that plays R (tests/tools/glue_driver.cpp).

CPU: the package layout, the exported signature, that the Makevars link line resolves every
symbol.  GPU: `set.seed(1234); bn_mcmc(network$data, network$dag_info, N = 50000)` -- R's stream
state goes in through .Random.seed, the trace equals the reference's (golden cfg1, the README
run) and the .Random.seed left behind equals R's state after the reference's 250,277 draws
(src/RcppExports.cpp:11-28)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GLUE_DIR = os.path.join(ROOT, "bayesnetworks_b200", "csrc", "rcpp_glue")
INT_COLS = ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP")


def makevars():
    """PKG_CPPFLAGS / PKG_LIBS of the glue's Makevars with BN_B200_HOME = this checkout."""
    out = subprocess.check_output(
        ["make", "-s", "-f", os.path.join(GLUE_DIR, "Makevars"), "-f", "/dev/stdin", f"BN_B200_HOME={ROOT}", "show"],
        input=b"show:\n\t@echo $(PKG_CPPFLAGS)\n\t@echo $(PKG_LIBS)\n")
    cpp, libs = out.decode().strip().split("\n")
    return cpp.split(), libs.split()


@pytest.fixture(scope="module")
def glue_so(tmp_path_factory):
    from bayesnetworks_b200 import build
    build.build()
    cpp, libs = makevars()
    so = str(tmp_path_factory.mktemp("glue") / "bayesnetworks_glue.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-w", "-fPIC", "-shared", "-Wl,--no-undefined",
                           f"-I{os.path.join(ROOT, 'oracle', 'ref_shim')}", f"-I{GLUE_DIR}"] + cpp +
                          ["-o", so, os.path.join(ROOT, "tests", "tools", "glue_driver.cpp")] + libs)
    return so


def test_package_layout_and_signature():
    """What the maintainer copies into src/: the replacement bayesnet_mcmc.cpp and a Makevars, both
    files; the exported signature, defaults and column order of the reference are kept."""
    assert sorted(os.listdir(GLUE_DIR)) == ["Makevars", "bayesnet_mcmc.cpp"]
    text = open(os.path.join(GLUE_DIR, "bayesnet_mcmc.cpp")).read()
    for frag in ("// [[Rcpp::export]]", "DataFrame main_fun(NumericMatrix X,", "std::vector<int> graph_source,",
                 "std::vector<int> graph_target,", "std::vector<int> graph_node_labels,",
                 "std::vector<int> graph_node_type,", "int MaxPar = 50,", "const double phi = 1,",
                 "const double omega = 6.9,", "const int InitialNetwork = 2,", "const int drop = 0,",
                 "int N = 1000,", "int output = 10)"):
        assert frag in text, frag
    assert re.findall(r'Named\("(\w+)"\)', text) == ["iter", "ChangedNode", "movetype", "globalLL", "additions",
                                                    "deletions", "FN", "FP"]
    cpp, libs = makevars()
    assert f"-I{ROOT}/include" in cpp
    assert "-lbn_b200" in libs and any(x.startswith("-Wl,-rpath,") for x in libs)


def test_glue_builds_and_links_with_the_makevars_line(glue_so):
    """Every symbol the glue needs is resolved by the Makevars link line (-Wl,--no-undefined)."""
    syms = subprocess.check_output(["nm", "-D", "--undefined-only", glue_so]).decode()
    assert "bn_main_fun" in syms and "bn_last_error" in syms
    lib = C.CDLL(glue_so)
    assert hasattr(lib, "glue_main_fun")


def _call(lib, X, src, tgt, nt, max_par, N, output, random_seed, initial_network=2):
    Xf = np.asfortranarray(X)
    n, p = Xf.shape
    cap = (N + output - 1) // output + 1
    ints = {k: np.zeros(cap, np.int32) for k in INT_COLS}
    gll = np.zeros(cap)
    labels = np.arange(p, dtype=np.int32)
    rs_in = None if random_seed is None else np.ascontiguousarray(random_seed, dtype=np.int32)
    rs_out = np.zeros(626, np.int32)
    draws = C.c_long(0)
    err = C.create_string_buffer(512)
    ip, dp = C.POINTER(C.c_int), C.POINTER(C.c_double)
    i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
    src, tgt, nt = i32(src), i32(tgt), i32(nt)
    rows = lib.glue_main_fun(
        Xf.ctypes.data_as(dp), n, p, src.ctypes.data_as(ip), tgt.ctypes.data_as(ip), len(src),
        labels.ctypes.data_as(ip), nt.ctypes.data_as(ip), max_par, C.c_double(1.0), C.c_double(6.9),
        initial_network, 0, N, output, None if rs_in is None else rs_in.ctypes.data_as(ip), rs_out.ctypes.data_as(ip),
        cap, ints["iter"].ctypes.data_as(ip), ints["ChangedNode"].ctypes.data_as(ip),
        ints["movetype"].ctypes.data_as(ip), gll.ctypes.data_as(dp), ints["additions"].ctypes.data_as(ip),
        ints["deletions"].ctypes.data_as(ip), ints["FN"].ctypes.data_as(ip), ints["FP"].ctypes.data_as(ip),
        C.byref(draws), err, 512)
    return rows, {k: v[:max(rows, 0)] for k, v in ints.items()}, gll[:max(rows, 0)], rs_out, draws.value, err.value.decode()


def test_glue_reports_errors_as_r_errors(glue_so, dataset):
    """Without a CUDA device (here) the library's status becomes an R error through Rcpp::stop; on
    the GPU box a bad argument does."""
    lib = C.CDLL(glue_so)
    X, src, tgt, nt = dataset["X"], dataset["source"], dataset["target"], dataset["node_type"]
    rows, _, _, _, _, err = _call(lib, X, src, tgt, nt, 200, 100, 10, None)   # max_par > 64
    assert rows == -1 and "bayesnetworks (B200)" in err


@pytest.mark.gpu
def test_set_seed_1234_through_the_glue(glue_so, dataset, golden, oracle):
    lib = C.CDLL(glue_so)
    X, src, tgt, nt = dataset["X"], dataset["source"], dataset["target"], dataset["node_type"]
    seed_in = np.concatenate([[10403], oracle.rmt_state_after(1234, 0)]).astype(np.int32)  # set.seed(1234)
    rows, ints, gll, seed_out, r_draws, err = _call(lib, X, src, tgt, nt, 50, 50000, 100, seed_in)
    assert rows == 500, err
    for k in INT_COLS:
        assert np.array_equal(ints[k], golden[f"cfg1_{k}"]), k
    assert np.allclose(gll, golden["cfg1_globalLL"], rtol=1e-9, atol=1e-9 * 1000)
    assert r_draws == 0   # nothing drawn from R's generator on the host: the stream state crossed the boundary
    n_draws = int(golden["cfg1_uniforms"])
    assert n_draws == 250277
    want = np.concatenate([[10403], oracle.rmt_state_after(1234, n_draws)]).astype(np.int32)
    assert np.array_equal(seed_out, want)   # what PutRNGstate leaves after the reference's run


@pytest.mark.gpu
def test_glue_other_rng_kind_falls_back_to_one_draw(glue_so, dataset):
    """RNGkind() is not the Mersenne-Twister: the chain is seeded from one unif_rand() draw."""
    lib = C.CDLL(glue_so)
    X, src, tgt, nt = dataset["X"], dataset["source"], dataset["target"], dataset["node_type"]
    seed_in = np.zeros(626, np.int32)
    seed_in[0] = 10407   # kind 7 (user-supplied); anything but %% 100 == 3
    rows, ints, gll, seed_out, r_draws, err = _call(lib, X, src, tgt, nt, 8, 2000, 100, seed_in)
    assert rows == 20 and r_draws == 1, err
