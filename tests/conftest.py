import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

os.environ.setdefault("MASTER_ADDR", "127.0.0.1")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (select with -m gpu)")


def pytest_collection_modifyitems(config, items):
    # `-m gpu` tests are skipped automatically where no CUDA device exists, so a plain `pytest tests/`
    # on a machine without a GPU never tries to launch a kernel.
    try:
        import torch

        has_cuda = torch.cuda.is_available()
    except Exception:
        has_cuda = False
    if has_cuda:
        return
    skip = pytest.mark.skip(reason="no CUDA device on this machine")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def _ref_recordings():
    """Tapes recorded in this session (RLB_RECORD_TAPES=DIR), written to DIR/<module>/<test function>.npz at the end."""
    import _ref_tape

    tapes = {}
    yield tapes
    for (module, function), ts in tapes.items():
        _ref_tape.save(_ref_tape.record_dir(), module, function, ts)


@pytest.fixture()
def _ref_tape(request, _ref_recordings):
    """This test's conversation with the reference: recorded live, or played back from tests/golden."""
    import _ref_tape

    module, function = request.node.module.__name__.rsplit(".", 1)[-1], request.node.originalname
    name = request.node.name
    if _ref_tape.record_dir() is not None:
        tape = _ref_tape.recorder(name)
        yield tape
        _ref_recordings.setdefault((module, function), []).append(tape)
        return
    tape = _ref_tape.player(module, function, name)
    yield tape
    assert tape.pos == len(tape.events), f"{name}: {len(tape.events) - tape.pos} recorded reference operations not replayed"


def _live_reference(tape, what: str):
    """The live reference object to record against; None on playback."""
    if not tape.recording:
        return None
    from oracle import ref_loader

    root = os.environ.get("RLB_REFERENCE_ROOT")
    if what in ("cpu", "cuda"):
        live = ref_loader.reference_ext(what)
    elif root is None:
        live = None
    else:
        live = ref_loader.reference_functionals(root) if what == "funcs" else ref_loader.reference_samplers(root)
    if live is None or (what == "cuda" and not hasattr(live, "CudaSumSegmentTreeFp32")):
        pytest.fail(f"recording needs the reference ({what}): set RLB_REFERENCE_ROOT and build oracle/_ref")
    return live


@pytest.fixture()
def ref_cpu(_ref_tape):
    """The compiled, unmodified reference CPU segment trees (SumSegmentTreeFp32, MinSegmentTreeFp32), recorded."""
    import _ref_tape as rt

    return rt.root(_ref_tape, "cpu", _live_reference(_ref_tape, "cpu"))


@pytest.fixture()
def ref_cuda(_ref_tape):
    """The compiled, unmodified reference CUDA segment trees (CudaSumSegmentTreeFp32, ...), recorded."""
    import _ref_tape as rt

    return rt.root(_ref_tape, "cuda", _live_reference(_ref_tape, "cuda"))


@pytest.fixture()
def ref_funcs(_ref_tape):
    """The reference's Python value functionals, recorded."""
    import _ref_tape as rt

    return rt.root(_ref_tape, "funcs", _live_reference(_ref_tape, "funcs"))


@pytest.fixture()
def ref_samplers(_ref_tape):
    """The reference's samplers module, unmodified, under stub imports (``.mod``, ``.make_storage``), recorded."""
    import _ref_tape as rt

    return rt.root(_ref_tape, "samplers", _live_reference(_ref_tape, "samplers"))


@pytest.fixture()
def emul():
    """Install the oracle-backed emulator as rl_b200's backend for one CPU host-logic test."""
    from rl_b200 import ops

    from _emul import OracleBackend

    ops.set_backend(OracleBackend())
    try:
        yield
    finally:
        ops.set_backend(None)


@pytest.fixture(scope="session")
def cuda_backend():
    """The real library on a real GPU (-m gpu tests)."""
    import torch

    from rl_b200 import ops

    assert torch.cuda.is_available()
    ops.set_backend(None)
    return ops.backend()
