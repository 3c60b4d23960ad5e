import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def pytest_collection_modifyitems(config, items):
    # On the GPU box a kernel that never finishes blocks the test process inside a CUDA call for good (and whatever was
    # to run after the tests with it). Every GPU test gets a bound; method "thread" = a watchdog thread that ends the
    # process, because a signal handler cannot interrupt a blocking C call. Not under the CPU emulation (CLDN_B200_LIB
    # set), whose sanitizer builds are slow by design.
    if os.environ.get("CLDN_B200_LIB"):
        return
    try:
        import pytest_timeout  # noqa: F401
    except ImportError:
        return
    for item in items:
        if item.get_closest_marker("gpu") and not item.get_closest_marker("timeout"):
            item.add_marker(pytest.mark.timeout(900, method="thread"))


@pytest.fixture(scope="session")
def lib_built():
    """The C-ABI library, built once per session (nvcc cross-compiles sm_100a without a GPU)."""
    from cloudini_b200 import build
    return build.build()


@pytest.fixture(scope="session")
def port(lib_built):
    from oracle.client import PortOracle
    return PortOracle()


@pytest.fixture(scope="session")
def ref(lib_built):
    """The compiled reference where it can be built, else its answers recorded in tests/golden/ref_answers.npz."""
    from oracle.client import RecordingRef, build_ref, reference_oracle
    build_ref()
    r = reference_oracle()
    yield r
    if isinstance(r, RecordingRef):
        r.save()


@pytest.fixture(scope="session")
def oracle(lib_built):
    """Best available checker: the compiled reference when present, else the C port (itself pinned by test_oracle.py)."""
    from oracle.client import best_oracle, build_ref
    build_ref()
    return best_oracle()


@pytest.fixture(scope="session")
def golden(lib_built):
    import cloudini_b200 as cb
    out = {}
    for fname in ("golden_v1.npz", "golden_v2.npz"):  # v2: the lossless float coders (XOR / Gorilla)
        z = np.load(os.path.join(ROOT, "tests", "golden", fname))
        for n in sorted({k.split("__")[0] for k in z.files}):
            info = cb.EncodingInfoFromYAML(bytes(z[n + "__yaml"]).decode())
            info.version = int(z[n + "__version"][0])
            info.use_threads = False
            out[n] = (info, z[n + "__input"], bytes(z[n + "__blob"]))
    return out


@pytest.fixture(scope="session")
def golden_ros(lib_built):
    """DDS messages + what the reference's converter made of them (tests/golden/make_golden_ros.py)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "golden_ros_v1.npz"))
    out = {}
    for n in sorted({k.split("__")[0] for k in z.files if not k.startswith("VIZ_")}):
        text = bytes(z[n + "__profile"]).decode()
        profile = {kv.split("=")[0]: float(kv.split("=")[1]) for kv in text.split(";") if kv}
        out[n] = {"msg": bytes(z[n + "__msg"]), "profile": profile, "default_resolution": float(z[n + "__opts"][0]),
                  "viz": bool(z[n + "__opts"][1]), "describe": bytes(z[n + "__describe"]).decode(),
                  "compressed": bytes(z[n + "__compressed"]), "restored": bytes(z[n + "__restored"])}
    return out


@pytest.fixture(scope="session")
def golden_viz(lib_built):
    """Raw clouds + what the reference's applyVizLossyPreprocessing made of them (tests/golden/make_golden_ros.py)."""
    import cloudini_b200 as cb
    z = np.load(os.path.join(ROOT, "tests", "golden", "golden_ros_v1.npz"))
    out = {}
    for n in sorted({k.split("__")[0] for k in z.files if k.startswith("VIZ_")}):
        info = cb.EncodingInfoFromYAML(bytes(z[n + "__yaml"]).decode())
        after = cb.EncodingInfoFromYAML(bytes(z[n + "__yaml_after"]).decode())
        out[n[4:]] = (info, z[n + "__input"], after, z[n + "__output"])
    return out
