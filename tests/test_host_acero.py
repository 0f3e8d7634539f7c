"""The Acero plug-in point (host/bkgpu_acero.hpp): a `bkgpu_fragment` exec node registered in Acero's factory registry the way the reference
registers its own nodes (src/exec/arrow_exec_node.cpp:444-477).  CPU: registration (and the refusal of a second one), the factory accepts
a fragment the library lowers and refuses one it does not (NotImplemented — the caller keeps its CPU declarations), and WITHOUT a GPU the
plan fails with the library's "no CPU fallback" message instead of computing anything.  GPU: record_batch_source -> bkgpu_fragment over a
table cut into small batches equals the oracle."""
import os
import subprocess

import pyarrow as pa
import pytest

from baikaldb_b200 import arrow_io, datagen, queries
from oracle import oracle
from tests.util import assert_same_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "baikaldb_b200", "bkgpu_acero_host")


@pytest.fixture(scope="module")
def acero_bin():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "host"), "acero", "PYARROW_DIR=" + os.path.dirname(pa.__file__)])
    return BIN


def _files(tmp_path, plan, cols, want):
    s, d = arrow_io.encode(cols)
    os_, _ = arrow_io.encode(want.columns)   # the fragment's output schema: "<tuple>_<slot>" fields typed by the Chunk map
    (tmp_path / "p").write_bytes(plan.serialize()); (tmp_path / "s").write_bytes(s); (tmp_path / "d").write_bytes(d); (tmp_path / "os").write_bytes(os_)
    return [str(tmp_path / x) for x in ("p", "s", "d", "os", "so", "do")]


def test_factory_registers_and_checks_the_fragment_on_the_host(acero_bin, tmp_path):
    (tmp_path / "p").write_bytes(queries.c2_filter_groupby().serialize())
    r = subprocess.run([acero_bin, "check", str(tmp_path / "p")], capture_output=True, text=True)
    assert r.returncode == 0 and "BkgpuFragmentNode" in r.stdout, r.stderr
    (tmp_path / "bad").write_bytes(b"\x00" * 24)
    r = subprocess.run([acero_bin, "check", str(tmp_path / "bad")], capture_output=True, text=True)
    assert r.returncode == 4 and "NotImplemented" in r.stderr and "does not take this fragment" in r.stderr


def test_without_a_gpu_the_plan_fails_loudly(acero_bin, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    cols = datagen.c2_table(0, 3000, n_groups=7)
    plan = queries.c2_filter_groupby()
    want = oracle.execute(plan.serialize(), cols)
    r = subprocess.run([acero_bin, "exec"] + _files(tmp_path, plan, cols, want), capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr, (r.returncode, r.stderr)
    assert not (tmp_path / "so").exists()


@pytest.mark.gpu
@pytest.mark.parametrize("batch_rows", [7000, 1 << 20])
def test_acero_plan_with_the_gpu_fragment_equals_the_oracle(acero_bin, tmp_path, batch_rows):
    cols = datagen.c2_table(0, 200_000, n_groups=77)
    plan = queries.c2_filter_groupby()
    want = oracle.execute(plan.serialize(), cols)
    r = subprocess.run([acero_bin, "exec"] + _files(tmp_path, plan, cols, want) + [str(batch_rows)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = arrow_io.decode((tmp_path / "so").read_bytes(), (tmp_path / "do").read_bytes(), plan.tuples)
    assert_same_rows(got, want.columns, ["0_1"])
