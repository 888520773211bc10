"""Cross-implementation parity on the GPU: the SAME oracle keys and inputs go
through this engine (in its own process, via the C-ABI harness of
tests/ref_cuda_runner.py) and are compared with what the reference's own CUDA
backend computed on them.  The reference's side is stored in
tests/golden/ref_cuda_parity_v1.npz, recorded once on a B200 by
tests/golden/make_ref_cuda_golden.py from the reference backend built
unmodified for sm_100 (oracle/build_ref_cuda.sh).  Asserted:
  * the keys and inputs are the ones the golden data was recorded on;
  * keyswitch: ours, the oracle and the reference agree on every word
    (the reference's output is pinned by its SHA-256);
  * PBS: our outputs and the reference's decrypt to f(m) on every sample, and
    our measured output-noise variance is at most twice the reference kernel's
    (the reference's own cross-backend criterion, core_crypto/gpu/algorithms/test/*.rs);
  * the phase error of our outputs is centred (no bias against the reference)."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_cuda_parity_v1.npz")
SEED = 0xB2000001
CASES = [("PARAM_MESSAGE_2_CARRY_2_KS_PBS", 192),
         ("PARAM_MULTI_BIT_GROUP_3_MESSAGE_2_CARRY_2_KS_PBS", 64),
         ("PARAM_GPU_MULTI_BIT_GROUP_4_MESSAGE_2_CARRY_2_KS_PBS", 64)]


def params(O, pname):
    from oracle import csprng

    return getattr(O, pname, None) or getattr(csprng, pname)


def case_inputs(O, keys, count):
    """The runner's input arrays for `count` samples, and the expected f(m)."""
    P = keys.params
    p = 16
    msgs = np.arange(count) % p
    f = [(5 * i + 3) % p for i in range(p)]
    big = O.lwe_encrypt_batch(O.Rng(31), keys.glwe_sk, msgs.astype(np.uint64) * np.uint64(P.delta), P.lwe_noise_log2)
    arrays = dict(bsk=keys.bsk, ksk=keys.ksk, big=big, lut=O.make_lut(P, f),
                  params=np.array([P.n, P.k, P.N, P.pbs_base_log, P.pbs_level, P.ks_base_log, P.ks_level,
                                   P.grouping_factor, int(P.centered_ms)]))
    return arrays, np.array([f[m] for m in msgs])


def sha256(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def run_lib(lib, inp, out):
    """KS -> PBS of the arrays in `inp` through one library in its own process."""
    env = dict(os.environ)
    env.pop("B200_LIB_PATH", None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "ref_cuda_runner.py"), "--lib", lib, "--inp", inp,
                        "--out", out], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return np.load(out)


@pytest.mark.parametrize("pname,count", CASES)
def test_same_keys_through_both_libraries(oracle, keyset, tmp_path, pname, count):
    O = oracle
    P = params(O, pname)
    keys = keyset(P, seed=SEED)
    arrays, want = case_inputs(O, keys, count)
    golden = np.load(GOLDEN)
    assert sha256(*arrays.values()) == str(golden[pname + "__inputs_sha256"]), \
        "keys / inputs differ from those the reference outputs were recorded on"
    inp = str(tmp_path / "in.npz")
    np.savez(inp, **arrays)
    ours = run_lib("ours", inp, str(tmp_path / "ours.npz"))
    want_small = O.keyswitch_batch(keys, arrays["big"])
    assert np.array_equal(ours["small"], want_small), "our keyswitch differs from the oracle"
    assert sha256(want_small) == str(golden[pname + "__ref_small_sha256"]), \
        "the reference's CUDA keyswitch differs from the oracle"
    p = 16
    err = {}
    for name, pt in (("ours", O.lwe_decrypt_batch(keys.glwe_sk, ours["out"])), ("ref", golden[pname + "__ref_phase"])):
        assert np.array_equal(O.decode(pt, P.delta, p), want), f"{name}: PBS outputs do not decrypt to f(m)"
        e = (pt - want.astype(np.uint64) * np.uint64(P.delta)).astype(np.int64).astype(np.float64) / 2.0 ** 64
        err[name] = e
    v_ours, v_ref = float(np.var(err["ours"])), float(np.var(err["ref"]))
    # ours may be quieter (the multi-bit register kernels round decomposition ties to even), never much louder
    assert v_ours < 2.0 * v_ref, (v_ours, v_ref)
    # (the output WORDS of the two are unrelated: any f64 rounding difference flips a decomposition digit and the
    #  masks then diverge chaotically -- equality is defined on the phase, as the reference does across backends)
    assert abs(float(np.mean(err["ours"]))) < 6.0 * np.sqrt(v_ours / count) + 2.0 ** -20
