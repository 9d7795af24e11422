"""CPU-only: every header of the CUDA library compiles as the only include of a translation unit (sm_100a, no GPU needed),
so no header depends on the include order of orbx.cu."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rgbd_visualodometry_b200", "csrc")
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    return nvcc if os.path.exists(nvcc) else None


@pytest.mark.parametrize("header", HEADERS)
def test_header_compiles_alone(header, tmp_path):
    nvcc = _nvcc()
    if not nvcc:
        pytest.skip("nvcc not available")
    src = tmp_path / "only.cu"
    src.write_text(f'#include "{os.path.join(CSRC, header)}"\n')
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-diag-suppress", "68", "-c",
                          "-o", str(tmp_path / "only.o"), str(src)], cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, f"{header} does not compile on its own:\n{out.stdout}{out.stderr}"
