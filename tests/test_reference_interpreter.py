"""The reference's own leaf functions under MATLAB / GNU Octave, when an interpreter AND the reference tree are present
(SURVEY.md section 8c: the only route from "parity unpinned" to pinned for everything beyond estimateTransform).

The reference's .m files are not part of this repository: PCREG_REFERENCE_DIR names a checkout of them.  Without it, or
without an interpreter (probed: matlab, octave, octave-cli), these tests SKIP with the reason printed.  Where both exist
they run the UNMODIFIED .m files (quickTF.m, invertTF.m, estimateTransform.m, getLocalPoints.m, AlignPoints.m,
AlignPoints_KNN.m, AlignPoints_weighted.m -- the last three need `pca` from the statistics package) on seeded inputs
exchanged as text files, and compare the oracle restatement (CPU test) and the CUDA path (gpu test) with what the
interpreter returned."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import oracle
from pcreg_b200 import synth

REF = os.environ.get("PCREG_REFERENCE_DIR", "")


def _interpreter():
    for exe in ("octave-cli", "octave", "matlab"):
        p = shutil.which(exe)
        if p:
            return exe, p
    return None, None


def _need():
    exe, path = _interpreter()
    if not path:
        pytest.skip("no MATLAB / Octave interpreter on this host (probed: octave-cli, octave, matlab)")
    if not REF or not os.path.isfile(os.path.join(REF, "estimateTransform.m")):
        pytest.skip("no reference tree: set PCREG_REFERENCE_DIR to a checkout of the reference's .m files")
    return exe, path


def _run(exe, path, script, cwd):
    if exe == "matlab":
        cmd = [path, "-batch", script]
    else:
        cmd = [path, "--no-gui", "--quiet", "--eval", "pkg load statistics; " + script] if _has_stats(path) else [path, "--no-gui", "--quiet", "--eval", script]
    r = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True, timeout=600)
    if r.returncode != 0:
        pytest.skip("interpreter failed on the reference leaf (missing toolbox?): %s" % (r.stderr.strip()[-300:] or r.stdout.strip()[-300:]))


def _has_stats(path):
    r = subprocess.run([path, "--no-gui", "--quiet", "--eval", "pkg load statistics"], capture_output=True, text=True, timeout=120)
    return r.returncode == 0


def _leafs(exe, path):
    """Runs the reference leafs once; returns dict name -> arrays."""
    g = synth.rng(31)
    d = tempfile.mkdtemp(prefix="pcreg_ref_")
    pts = g.normal(0, 3, (400, 3)) @ np.diag([3.0, 1.5, 0.4]) + np.array([5.0, -2.0, 9.0])
    T = synth.make_T(synth.rot_xyz([0.3, -0.7, 1.9]), np.array([13.0, 25.0, -17.0]))
    p2 = g.normal(0, 10, (60, 3))
    p1 = synth.apply_T(p2, T) + g.normal(0, 0.01, (60, 3))
    cloud = g.uniform(0, 10, (5000, 3))
    for name, a in (("pts", pts), ("T", T), ("p1", p1), ("p2", p2), ("cloud", cloud)):
        np.savetxt(os.path.join(d, name + ".txt"), a, fmt="%.17g")
    wr = lambda v: "dlmwrite('%s.txt', %s, 'delimiter', ' ', 'precision', '%%.17g'); " % (v, v)
    script = ("addpath('%s'); pts = load('pts.txt'); T = load('T.txt'); p1 = load('p1.txt'); p2 = load('p2.txt'); cloud = load('cloud.txt'); "
              "q = quickTF(pts, T); Ti = invertTF(T); Te = estimateTransform(p1, p2); "
              "[lp, ld] = getLocalPoints(cloud, 2.5, [3 3 3], 10, 100000); " % REF) + wr("q") + wr("Ti") + wr("Te") + wr("lp") + wr("ld")
    _run(exe, path, script, d)
    out = dict(pts=pts, T=T, p1=p1, p2=p2, cloud=cloud)
    for v in ("q", "Ti", "Te", "lp", "ld"):
        out[v] = np.loadtxt(os.path.join(d, v + ".txt"), ndmin=2)
    # the AlignPoints family needs pca (statistics package / toolbox): separate run, optional
    script2 = ("addpath('%s'); pts = load('pts.txt'); [a1, c1] = AlignPoints(pts); [a2, c2, m2] = AlignPoints_KNN(pts); "
               "[a4, c4] = AlignPoints_weighted(pts); " % REF) + wr("a1") + wr("c1") + wr("a2") + wr("c2") + wr("a4") + wr("c4")
    try:
        _run(exe, path, script2, d)
        for v in ("a1", "c1", "a2", "c2", "a4", "c4"):
            out[v] = np.loadtxt(os.path.join(d, v + ".txt"), ndmin=2)
    except BaseException:                                   # pytest.skip raises: the family stays unchecked
        pass
    return out


def test_oracle_matches_reference_leafs_under_the_interpreter():
    exe, path = _need()
    R = _leafs(exe, path)
    np.testing.assert_allclose(oracle.quickTF(R["pts"], R["T"]), R["q"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(oracle.invertTF(R["T"]), R["Ti"], rtol=0, atol=1e-13)
    np.testing.assert_allclose(oracle.estimateTransform(R["p1"], R["p2"]), R["Te"], rtol=0, atol=1e-9)
    lp, ld = oracle.getLocalPoints(R["cloud"], 2.5, np.array([3.0, 3.0, 3.0]), 10, 100000)
    np.testing.assert_allclose(lp, R["lp"], atol=1e-13)
    np.testing.assert_allclose(np.ravel(ld), np.ravel(R["ld"]), atol=1e-13)
    if "a1" in R:
        a, c = oracle.AlignPoints(R["pts"])
        np.testing.assert_allclose(a, R["a1"], atol=1e-9)
        a, c, _ = oracle.AlignPoints_KNN(R["pts"])
        np.testing.assert_allclose(a, R["a2"], atol=1e-9)


@pytest.mark.gpu
def test_cuda_matches_reference_leafs_under_the_interpreter(pcreg):
    exe, path = _need()
    R = _leafs(exe, path)
    np.testing.assert_allclose(pcreg.quickTF(R["pts"], R["T"]), R["q"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(pcreg.estimateTransform(R["p1"], R["p2"]), R["Te"], rtol=0, atol=1e-9)
    if "a1" in R:
        a, c = pcreg.AlignPoints(R["pts"])
        np.testing.assert_allclose(a, R["a1"], atol=1e-9)
        a, c, _ = pcreg.AlignPoints_KNN(R["pts"])
        np.testing.assert_allclose(a, R["a2"], atol=1e-9)
        a, c = pcreg.AlignPoints_weighted(R["pts"])
        np.testing.assert_allclose(np.abs(a), np.abs(R["a4"]), atol=1e-9)      # column order of eig(M) is unpinned: compare up to permutation sign
