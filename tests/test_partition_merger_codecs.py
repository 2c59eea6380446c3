"""ObGpuPartitionMajorMerger::write_column_groups with per-column encodings (tests/cpp/test_partition_merger_codecs.cpp): built by
__graft_entry__.build(); without a device the adapter refuses (exit 77), with one every group equals the host writer's image of
the oracle's merged rows with the same encodings."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "test_partition_merger_codecs")


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_codec_merger_builds_and_refuses_without_device():
    assert os.path.exists(BIN)
    if _has_gpu():
        pytest.skip("device present: covered by the gpu test")
    r = subprocess.run([BIN], capture_output=True, text=True, timeout=120)
    assert r.returncode == 77, r.stdout + r.stderr


@pytest.mark.gpu
def test_codec_merger_parity_on_gpu():
    r = subprocess.run([BIN], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert "partition merger codec tests passed" in r.stdout
