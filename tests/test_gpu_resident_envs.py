"""resident_envs(): one resident wave of the two-term runner (k_run<NV, false, true>), which keeps more warps on an SM than
the general runner; and the general runner on a handle of that many slots, which exceeds its own wave."""
import ctypes as C

import pytest

from test_gpu_parity import RECORD_FIELDS, assert_records_equal, reference_records

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def runner_wave(torch, nv, two):
    """Resident warps of k_run<nv, false, two> on device 0, from the CUDA runtime's occupancy calculator and the block
    size the kernel's launch bounds state (cudaFuncAttributes::maxThreadsPerBlock)."""
    from deepgroebner_b200 import _lib
    lib = _lib.load()
    cudart = C.CDLL("libcudart.so.12")   # the runtime libbbenv.so registered its kernels with
    stub = C.cast(getattr(lib, "_Z5k_runILi%dELb0ELb%dEEv8BBParamsS0_9BBRunArgs" % (nv, int(two))), C.c_void_p)
    attr = (C.c_char * 512)()   # cudaFuncAttributes: three size_t, then maxThreadsPerBlock
    assert cudart.cudaFuncGetAttributes(attr, stub) == 0
    threads = C.c_int.from_buffer(attr, 3 * C.sizeof(C.c_size_t)).value
    blocks = C.c_int(0)
    assert cudart.cudaOccupancyMaxActiveBlocksPerMultiprocessor(C.byref(blocks), stub, threads, C.c_size_t(0)) == 0
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return sms * blocks.value * (threads // 32)


@pytest.mark.parametrize("nv", [3, 5])
def test_resident_envs_is_the_two_term_runners_wave(torch_cuda, nv):
    from deepgroebner_b200.buchberger import resident_envs
    n = resident_envs(0, nv)   # also sets the runners' shared-memory carveout, which the occupancy depends on
    two, general = runner_wave(torch_cuda, nv, True), runner_wave(torch_cuda, nv, False)
    assert n == two > general, (n, two, general)


def test_general_runner_on_a_two_term_sized_handle(torch_cuda):
    """bench.py sizes its handle with resident_envs(); forced through the general runner, whose wave is smaller, the
    16384 episodes of 3-20-10-weighted under Degree still equal the reference's records, and the counters add up."""
    from deepgroebner_b200.buchberger import BuchbergerEngine, resident_envs
    slots = resident_envs(0, 3)
    assert slots > runner_wave(torch_cuda, 3, False)
    eng = BuchbergerEngine("3-20-10-weighted", num_envs=slots)
    eng.set_two_term(False)
    eng.counters(reset=True)
    s, _ = eng.run_episodes("degree", episodes=16384, seed_base=0, compute_gb=True)
    c = eng.counters(reset=True)
    assert (s["status"] == 2).all()
    assert c["episodes"] == 16384 and c["env_steps"] == int(s["steps"].sum()) and c["additions"] == int(s["additions"].sum())
    assert_records_equal(s, reference_records("3-20-10-weighted", "degree", 16384), "general runner, %d slots" % slots)
    eng.set_two_term(True)
    t, _ = eng.run_episodes("degree", episodes=16384, seed_base=0, compute_gb=True)
    for f in RECORD_FIELDS:
        assert (t[f] == s[f]).all(), f
