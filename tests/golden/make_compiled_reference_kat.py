#!/usr/bin/env python3
"""Regenerate tests/golden/compiled_reference_kat.json: the answers of the reference's own code, compiled
unchanged into oracle/_ref by oracle/Makefile (needs the reference checkout at build time), on the inputs
of tests/helpers.py (compiled_reference_keccak_messages, compiled_reference_secure_tries).

  keccak       ethash/lib/keccak/keccak.c          ethash_keccak256 of every message
  secure_trie  evmone/test/state/mpt.cpp           root of every trie (through oracle/ref_shim.cpp)

tests/test_oracle_golden.py compares the oracle's port with these answers, so the comparison runs on
machines without the reference.
"""
import ctypes as C
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib  # noqa: E402
from helpers import compiled_reference_keccak_messages, compiled_reference_secure_tries, inputs_sha256  # noqa: E402


def main():
    for path in (oracle_lib.REF_KECCAK_PATH, oracle_lib.REF_EVMONE_PATH):
        if not os.path.exists(path):
            sys.exit(f"{path} missing: run `make -C oracle` where the reference checkout is present")
    o = oracle_lib.get()
    msgs = compiled_reference_keccak_messages()
    keccak = [{"len": len(m), "keccak256": o.ref_keccak256(m).hex()} for m in msgs]
    ref = C.CDLL(oracle_lib.REF_EVMONE_PATH)
    tries = compiled_reference_secure_tries()
    secure = []
    for kv in tries:
        k, koff = oracle_lib.csr([a for a, _ in kv], np.uint32)
        v, voff = oracle_lib.csr([b for _, b in kv], np.uint64)
        out = np.zeros(32, np.uint8)
        ref.ref_evmone_mpt_root(k.ctypes.data_as(oracle_lib.u8p), koff.ctypes.data_as(oracle_lib.u32p),
                                v.ctypes.data_as(oracle_lib.u8p), voff.ctypes.data_as(oracle_lib.u64p), C.c_uint64(len(kv)),
                                out.ctypes.data_as(oracle_lib.u8p))
        secure.append({"n": len(kv), "root": out.tobytes().hex()})
    doc = {"source": "oracle/_ref: ethash/lib/keccak/keccak.c and evmone/test/state/mpt.cpp compiled unchanged (oracle/Makefile)",
           "keccak": keccak, "keccak_inputs_sha256": inputs_sha256(msgs),
           "secure_trie": secure, "secure_trie_inputs_sha256": inputs_sha256([a + b for kv in tries for a, b in kv])}
    path = os.path.join(HERE, "compiled_reference_kat.json")
    with open(path, "w") as f:
        f.write(json.dumps(doc, separators=(",", ":"), sort_keys=True) + "\n")
    print(f"compiled_reference_kat.json: {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
