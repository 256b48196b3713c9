"""The MEX gateway of the pose covariance (pcreg_b200/csrc/pcreg_mex_cov.cpp) without MATLAB: type-checked against the stand-in
mex.h, every ABI symbol it calls declared in include/pcreg.h, and its marshaling executed against the in-memory mx* runtime with a
stub of pcreg_icp_covariance (tests/fake_mex/cov_harness.cpp): offsets handed over as int64, optional ref / targets / w_src,
tre turned from [H][K] to H x K column-major, argument errors, no leaked arrays."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GATEWAY = os.path.join(ROOT, "pcreg_b200", "csrc", "pcreg_mex_cov.cpp")
FAKE = os.path.join(ROOT, "tests", "fake_mex")


def test_cov_gateway_typechecks_against_fake_mex():
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-Werror", "-I", FAKE, GATEWAY], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_cov_gateway_marshaling_runs_against_fake_runtime(tmp_path):
    exe = str(tmp_path / "cov_harness")
    r = subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-I", FAKE, os.path.join(FAKE, "cov_harness.cpp"), GATEWAY, "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("OK:"), r.stdout + r.stderr


def test_cov_gateway_only_calls_declared_abi():
    with open(os.path.join(ROOT, "include", "pcreg.h")) as f:
        hdr = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    declared = set(re.findall(r"\b(pcreg_[a-z0-9_]+)\s*\(", hdr))
    used = set()
    for name in ("pcreg_mex_cov.cpp", "pcreg_mex_util.h"):
        with open(os.path.join(ROOT, "pcreg_b200", "csrc", name)) as f:
            used |= set(re.findall(r"\b(pcreg_[a-z0-9_]+)\s*\(", re.sub(r"//.*", "", f.read())))
    used -= {"pcreg_mex_cov"}
    assert "pcreg_icp_covariance" in used and used <= declared, used - declared


def test_cov_shim_calls_the_gateway():
    with open(os.path.join(ROOT, "pcreg_b200", "matlab", "pcreg_icp_cov.m")) as f:
        text = f.read()
    assert text.startswith("function") and "pcreg_icp_cov(" in text.splitlines()[0] and "pcreg_mex_cov(" in text
