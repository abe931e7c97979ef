import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def cpu():
    """Our C restatement of the reference (oracle/cpu_ref.c)."""
    from oracle import oracle
    return oracle.cpu()


@pytest.fixture
def ref(request, cpu, isa):
    """The reference's own AVX2/SSE4 loops: oracle/_ref where it was built, otherwise their recorded
    replay (tests/ref_replay.py)."""
    import ref_replay
    from oracle import oracle
    lib = oracle.ref()
    key = ref_replay.key_of(request.node)
    if lib is None:
        replay = ref_replay.Replay(key, cpu)
        yield replay
        replay.done()
    elif os.environ.get(ref_replay.RECORD_ENV):
        yield ref_replay.Recorder(lib, key, cpu, isa)
    else:
        yield lib


@pytest.fixture(scope="session")
def isa():
    """The ISA whose reference loops the tests compare against: the host's, or the recorded one."""
    import ref_replay
    from oracle import oracle
    return oracle.host_isa() if oracle.ref() is not None else ref_replay.table()["isa"]


@pytest.fixture(scope="session")
def ag():
    """The product library through its C ABI.  GPU tests fail loudly if it cannot run."""
    from arrow_go_b200 import _native as N
    N.call("ag_init", -1)
    return N
