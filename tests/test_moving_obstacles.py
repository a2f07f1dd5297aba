"""CPU checks of the constant-velocity obstacle entry point (no GPU needed): the library reports ABI version 103 and
dsmppi_set_obstacle_velocities fails loudly on a null context.  The GPU behaviour is in
tests/test_gpu_moving_obstacles.py."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from optimalmodulationds_b200 import _capi, build
    build.build()
    return _capi.load()


def test_version_is_103(lib):
    assert lib.dsmppi_version() == 103


def test_set_obstacle_velocities_refuses_a_null_context(lib):
    lib.dsmppi_set_obstacles(None, None, 1, None)      # leave an unrelated message behind first
    before = lib.dsmppi_last_error()
    assert lib.dsmppi_set_obstacle_velocities(None, None, 1, None) != 0
    msg = lib.dsmppi_last_error()
    assert msg and b"ctx" in msg and msg != before
