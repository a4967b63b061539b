"""CPU check of the bit helpers of the fused multi-k sketch loop (tests/host/fused_bits_test.cpp); no GPU needed."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fused_bit_helpers(tmp_path):
    exe = str(tmp_path / "fused_bits_test")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe,
                           os.path.join(ROOT, "tests", "host", "fused_bits_test.cpp")])
    out = subprocess.run([exe], stdout=subprocess.PIPE, text=True)
    assert out.returncode == 0, out.stdout
