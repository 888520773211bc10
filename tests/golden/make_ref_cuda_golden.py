"""Record the reference CUDA backend's side of tests/test_ref_cuda_parity.py.

Needs a GPU and oracle/_ref/libtfhe_cuda_backend_ref.so, which
oracle/build_ref_cuda.sh builds from the reference's unmodified sources.  For
every case of the test, KS -> PBS runs through the reference library on the
test's keys and inputs; ref_cuda_parity_v1.npz then holds, per parameter set:
  <param>__inputs_sha256     digest of the keys / inputs given to the library
  <param>__ref_small_sha256  digest of the reference's keyswitched ciphertexts
  <param>__ref_phase         the reference's PBS outputs decrypted under the
                             oracle's GLWE key (what the noise comparison uses)
and `device`, the GPU the outputs were computed on.  Run:
    python tests/golden/make_ref_cuda_golden.py
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "ref_cuda_parity_v1.npz")


def main():
    import torch

    from oracle import oracle as O
    from tests.test_ref_cuda_parity import CASES, SEED, case_inputs, params, run_lib, sha256

    O.build()
    out = {"device": np.array(torch.cuda.get_device_name(0))}
    with tempfile.TemporaryDirectory() as tmp:
        for pname, count in CASES:
            keys = O.keygen(params(O, pname), SEED)
            arrays, want = case_inputs(O, keys, count)
            inp = os.path.join(tmp, "in.npz")
            np.savez(inp, **arrays)
            ref = run_lib("ref", inp, os.path.join(tmp, "ref.npz"))
            phase = O.lwe_decrypt_batch(keys.glwe_sk, ref["out"])
            out[pname + "__inputs_sha256"] = np.array(sha256(*arrays.values()))
            out[pname + "__ref_small_sha256"] = np.array(sha256(ref["small"]))
            out[pname + "__ref_phase"] = phase
            print(pname, "keyswitch == oracle:", np.array_equal(ref["small"], O.keyswitch_batch(keys, arrays["big"])),
                  "decrypts to f(m):", np.array_equal(O.decode(phase, keys.params.delta, 16), want))
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
