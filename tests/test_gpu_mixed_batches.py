"""-m gpu: the batched calls of managers that hold several model types (tests/cpp/mixed_batch_test.cpp).

A plain and a sharded manager holding uniform-acceleration, angular-rates and uniform-velocity targets with interleaved ids must
give, bit for bit, what one homogeneous manager per model type gives when it receives the records of its ids in call order:
updateBatch (ascending, shuffled, repeated and unknown ids, mixed actions), getEstimatesBatch, initBatch over ids of other types,
eraseBatch, watch / log, IntersectionSolver::query, nearestTargets and earliestIntersections.  The shards all live on device 0."""
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    lib = os.path.join(ROOT, "target_estimation_b200", "lib")
    path = str(tmp_path_factory.mktemp("mixed") / "mixed_batch_test")
    subprocess.check_call(["g++", "-O1", "-ffp-contract=off", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "mixed_batch_test.cpp"), "-o", path, "-L", lib, "-ltarget_c", "-lte_pool",
                           "-Wl,-rpath," + lib])
    return path


def _run(exe, *args):
    r = subprocess.run([exe, os.path.join(ROOT, "models")] + [str(a) for a in args], capture_output=True, text=True, timeout=900)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("ok:")


@pytest.mark.parametrize("shards", [1, 3])
def test_mixed_batches_match_one_manager_per_model_type(exe, shards):
    _run(exe, shards, "checks")


@pytest.mark.parametrize("shards", [1, 3])
def test_update_ops_without_measurements_raise_on_mixed_managers(exe, shards):
    """meas NULL with action NULL or with an UPDATE op raises before any pool is stepped, as on a homogeneous manager; a batch of
    predictions needs no measurements"""
    _run(exe, shards, "nomeas")
