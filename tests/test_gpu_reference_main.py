"""The drop-in boundary proven against the reference's OWN caller: oracle/_ref/miniVite_ref_gpu is the reference's
unmodified main.cpp (command line, GenerateRGG / file reader, timer brackets, report block) with exactly the patch
of INTEGRATION.md section 2 applied by oracle/build_ref.py --gpu -- distLouvainMethod (main.cpp:168-169) replaced by
mvgpu_upload_shard + mvgpu_louvain through the C ABI -- compiled against the MPI shim and linked with -lmvgpu.
Its traces must equal the goldens of the unpatched reference."""
import os

import pytest

from helpers import assert_trace_matches

pytestmark = pytest.mark.gpu


def _run(args, nranks=1):
    from oracle import oracle as O
    if not os.path.exists(O.REF_GPU_BIN):
        pytest.skip("oracle/_ref/miniVite_ref_gpu not built (needs the reference's sources at build time)")
    return O.run_reference(args, nranks=nranks, threads=2, trace=True, binary=O.REF_GPU_BIN, timeout=600)


def _check(r, case):
    assert r["result"]["iters"] == case["iters"]
    assert r["final"]["mod_repr"] == case["modularity"]
    assert repr(r["final"]["constant"]) == case["constant"]
    assert_trace_matches(case, r["result"]["iters"], r["final"]["modularity"], r["trace"], r["final"]["chash"])
    # the reference's own report block is still printed by its own code
    assert "Modularity, #Iterations:" in r["stdout"] and "64-bit datatype" in r["stdout"]


def test_reference_main_with_gpu_patch_single_rank(golden):
    from minivite_b200 import gpu as G
    if G.device_count() < 1:
        pytest.fail("no CUDA device visible")
    _check(_run(["-n", 16384]), golden["rgg_n16384_p1"])
    _check(_run(["-n", 65536]), golden["rgg_n65536_p1"])


def test_reference_main_with_gpu_patch_two_ranks(golden):
    from minivite_b200 import gpu as G
    if G.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _check(_run(["-n", 16384], nranks=2), golden["rgg_n16384_p2"])
