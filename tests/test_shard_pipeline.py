"""The ordered shard pipeline of the file drivers (csrc/host/shard_pipeline.hpp), with fake steps, under ThreadSanitizer and under
AddressSanitizer + UBSan."""
import os
import subprocess

import pytest

from conftest import ROOT


@pytest.mark.parametrize("sanitize", ["thread", "address,undefined"])
def test_shard_pipeline(tmp_path, sanitize):
    exe = str(tmp_path / "shard_pipeline")
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-pthread", "-fsanitize=" + sanitize, "-fno-sanitize-recover=all", "-Wall",
                    "-o", exe, os.path.join(ROOT, "tests", "units", "shard_pipeline.cpp")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "shard pipeline ok" in r.stdout
