"""The device header's permutation, compiled as HOST code (tests/hostcheck/keccak_header_host.cpp defines the CUDA
qualifiers and the two funnel-shift intrinsics away), against the oracle: pins the rho/pi/chi index tables and the
digest-only last round (keccak_last_round_digest) without a GPU.  The product never runs this way."""
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def test_device_header_permutation_on_host(oracle, tmp_path):
    exe = str(tmp_path / "kh")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", exe, os.path.join(HERE, "hostcheck", "keccak_header_host.cpp")], check=True)
    rng = np.random.default_rng(5)
    msgs = [bytes(rng.integers(0, 256, n, dtype=np.uint8)) for n in list(range(0, 300)) + [532, 543, 544, 545, 1000, 4096]]
    stdin = "\n".join(m.hex() if m else "-" for m in msgs) + "\n"
    out = subprocess.run([exe], input=stdin, capture_output=True, text=True, check=True).stdout.split("\n")
    for m, line in zip(msgs, out):
        full, digest_only = line.split()
        want = oracle.keccak256(m).hex()
        assert full == want, len(m)
        assert digest_only == want, len(m)


def test_staged_absorb_path_on_host(oracle, tmp_path):
    """the staged kernel's per-lane absorb path (window copy, byte skew, in-slot padding, masked fallback) as host code
    (tests/hostcheck/stage_host.cpp) for every length 0..700 at every byte skew 0..15, plus long messages: digests equal the
    oracle's, stale slot bytes (0xEE) and neighbouring message bytes (0xA5) never leak in, and the fallback is exercised;
    then the aligned absorb at the skews that allow it (0, 4, 8, 12)"""
    exe = str(tmp_path / "sh")
    subprocess.run(["g++", "-O1", "-std=c++17", "-Wno-unknown-pragmas", "-o", exe, os.path.join(HERE, "hostcheck", "stage_host.cpp")], check=True)
    rng = np.random.default_rng(6)
    cases = [(sk, bytes(rng.integers(0, 256, n, dtype=np.uint8))) for n in range(0, 701) for sk in range(16)]
    cases += [(int(rng.integers(0, 64)), bytes(rng.integers(0, 256, int(n), dtype=np.uint8))) for n in rng.integers(700, 6000, 200)]
    stdin = "".join(f"{sk} {m.hex() if m else '-'}\n" for sk, m in cases)
    r = subprocess.run([exe], input=stdin, capture_output=True, text=True, check=True)
    out = r.stdout.split("\n")
    memo = {}
    for (sk, m), got in zip(cases, out):
        want = memo.get(m)
        if want is None:
            want = memo[m] = oracle.keccak256(m).hex()
        assert got == want, (sk, len(m))
    fallbacks = int(r.stderr.split()[-1])
    assert 0 < fallbacks < len(cases) // 20  # exercised, and rare (only 544..559 bytes left in the window)
    # the aligned absorb (no funnel shifts), taken when every lane's message starts at a multiple of 4: skews 0, 4, 8, 12
    aligned = [(sk, m) for sk, m in cases if sk % 4 == 0]
    stdin = "".join(f"{sk} {m.hex() if m else '-'}\n" for sk, m in aligned)
    r = subprocess.run([exe, "aligned"], input=stdin, capture_output=True, text=True, check=True)
    for (sk, m), got in zip(aligned, r.stdout.split("\n")):
        assert got == memo[m], ("aligned", sk, len(m))
    assert len(r.stdout.split()) == len(aligned) and int(r.stderr.split()[-1]) > 0
