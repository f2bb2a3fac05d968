"""Bank-conflict freedom of every shared-memory exchange access of the 16-point ring kernel at N = 1024, 2048
and 4096 (tests/emu/emu_banks.cpp: the kernel's own index functions, run on the CPU)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ring_exchange_bank_conflicts(tmp_path):
    exe = str(tmp_path / "emu_banks")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "emu", "emu_banks.cpp")],
                   check=True)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "640 wavefronts per frame" in res.stdout
