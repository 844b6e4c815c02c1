"""The C-ABI library loads and exports every symbol include/ls_b200.h declares; host-only logic
(YAML chain reader, rigid-matrix check) works; and the product refuses to run without a GPU
(no CPU fallback).  No compute entry point is called here."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ls():
    import laser_slam_b200 as m
    m.build()
    return m


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "ls_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ls_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(ls):
    lib = ctypes.CDLL(ls.LIB_PATH)
    syms = declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/ls_b200.h but not exported"


REF_YAML = """
readingDataPointsFilters:
  - RandomSamplingDataPointsFilter:
      prob: 0.5
referenceDataPointsFilters:
  - SamplingSurfaceNormalDataPointsFilter:
      knn: 10
matcher:
  KDTreeMatcher:
    knn: 1
    epsilon: 0
outlierFilters:
  - TrimmedDistOutlierFilter:
      ratio: 0.75
errorMinimizer:
  PointToPlaneErrorMinimizer
transformationCheckers:
  - CounterTransformationChecker:
      maxIterationCount: 40
  - DifferentialTransformationChecker:
      minDiffRotErr: 0.001
      minDiffTransErr: 0.01
      smoothLength: 4
#inspector:
#  NullInspector
inspector:
 VTKFileInspector:
     baseFileName: pointmatcher-run1
logger:
  NullLogger
"""


def test_yaml_chain_reader(ls):
    ref_yaml = REF_YAML
    p = ls.params_from_yaml(ref_yaml)
    assert (p.max_iterations, p.use_differential, p.smooth_length) == (40, 1, 4)
    assert abs(p.trim_ratio - 0.75) < 1e-7 and abs(p.min_diff_rot - 1e-3) < 1e-9 and abs(p.min_diff_trans - 1e-2) < 1e-9
    p2 = ls.params_from_yaml(ref_yaml.replace("maxIterationCount: 40", "maxIterationCount: 7").replace("ratio: 0.75", "ratio: 0.9"))
    assert p2.max_iterations == 7 and abs(p2.trim_ratio - 0.9) < 1e-7
    p3 = ls.params_from_yaml("matcher:\n  KDTreeMatcher:\n    knn: 1\ntransformationCheckers:\n  - CounterTransformationChecker:\n      maxIterationCount: 30\n")
    assert p3.use_differential == 0 and p3.max_iterations == 30 and p3.trim_ratio == 1.0
    for bad in ("matcher:\n  KDTreeMatcher:\n    knn: 3\n", "matcher:\n  KDTreeMatcher:\n    epsilon: 0.5\n",
                "errorMinimizer:\n  PointToPointErrorMinimizer\n", "outlierFilters:\n  - MaxDistOutlierFilter:\n      maxDist: 1\n"):
        with pytest.raises(ls.LsError):
            ls.params_from_yaml(bad)


def test_reference_default_yaml_is_accepted(ls):
    """The reference's own chain file must parse: tests/golden/icp_default.yaml is a byte-for-byte copy of
    laser_slam/configurations/icp_default.yaml from ethz-asl/laser_slam (BSD-3-Clause)."""
    p = ls.params_from_yaml(open(os.path.join(ROOT, "tests", "golden", "icp_default.yaml")).read())
    assert p.max_iterations == 40 and p.use_differential == 1 and abs(p.trim_ratio - 0.75) < 1e-7


def test_rigid_helpers_match_oracle(ls, oracle_mod):
    rng = np.random.default_rng(0)
    for _ in range(20):
        T = np.eye(4, dtype=np.float32)
        T[:3, :3] += rng.normal(scale=0.02, size=(3, 3)).astype(np.float32)
        T[:3, 3] = rng.normal(size=3)
        assert ls.check_rigid(T) == oracle_mod.check_rigid(T)
        assert np.array_equal(ls.correct_rigid(T), oracle_mod.correct_rigid(T))


def test_no_gpu_means_loud_failure(ls):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ls.LsError, match="no usable CUDA device"):
        ls.Context(0)


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under laser_slam_b200/ may reference it."""
    pkg = os.path.join(ROOT, "laser_slam_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", text, flags=re.M), f
                assert not re.search(r"#\s*include\s*[\"<][^\">]*oracle", text), f
                assert "libls_oracle" not in text and "lso_" not in text, f


def test_yaml_reports_the_filter_sections_it_does_not_apply(ls):
    """icp_default.yaml:1-7: the reading / reference DataPointsFilters are parsed and reported (they run upstream of the
    registration: ls_keep_point, ls_estimate_normals), not silently dropped."""
    p = ls.params_from_yaml(REF_YAML)
    assert abs(p.reading_sampling_prob - 0.5) < 1e-7 and p.reference_normals_knn == 10
    assert p.reference_sampling_ratio == 1.0 and p.unapplied_modules == 2
    assert p.max_iterations == 40 and abs(p.trim_ratio - 0.75) < 1e-7 and p.use_differential == 1
    q = ls.default_params()
    assert q.reading_sampling_prob == 1.0 and q.reference_normals_knn == 0 and q.unapplied_modules == 0


def test_keep_point_matches_the_oracle_rule(ls):
    """ls_keep_point (deterministic RandomSamplingDataPointsFilter) == oracle.keep_mask, and keeps about `prob` of the points."""
    import oracle
    for salt, prob in ((ls.READING_SALT, 0.5), (ls.REFERENCE_SALT, 0.25), (3, 0.999), (4, 1.0), (5, 0.0)):
        got = ls.keep_mask(20000, salt, prob)
        want = oracle.keep_mask(20000, salt, prob)
        assert np.array_equal(got, want)
        assert abs(got.mean() - prob) < 0.02
    assert not np.array_equal(ls.keep_mask(5000, 1, 0.5), ls.keep_mask(5000, 2, 0.5))


def test_reference_call_sites_compile_against_the_headers():
    """SURVEY.md §8b: the members laser_slam_ros and laser_slam's own sources use compile against include/ (tests/compile)."""
    import subprocess
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++17", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "compile", "reference_call_sites.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_datapoints_copy_on_write_and_views(tmp_path):
    """The compat DataPoints: copies share storage until written, views borrow caller memory (tests/compile)."""
    import subprocess
    exe = str(tmp_path / "dp_storage")
    build = os.path.join(ROOT, "laser_slam_b200", "_build")
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "compile", "datapoints_storage.cpp"), "-o", exe,
                        "-L", build, "-lls_b200", f"-Wl,-rpath,{build}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr
