"""Pins the size queries of the caller-allocated buffers (saved-for-backward blobs and workspaces) to exact values.
Callers allocate with these queries and the library carves the buffers with the same layout structs, so a region added
to one without the other would go unnoticed by every other test.  Host-only functions: no GPU needed.

The shapes cover the benchmark's c2 config, c4's per-GPU shape, F not divisible by 4 (70), F not a multiple of 64
(772, 900), V not divisible by 4 (37) and B < 128."""
import pytest

DISC_SHAPES = [(256, 20, 64, 64, 900), (3, 7, 2, 2, 70), (5, 32, 64, 64, 772)]        # N, L, De, R, F


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from gic_b200 import _lib
    return _lib.lib()


@pytest.mark.parametrize("shape,want", zip(DISC_SHAPES, [41369600, 1376, 699200]))
def test_disc_saved_floats(lib, shape, want):
    assert lib.gic_disc_saved_floats(*shape) == want


@pytest.mark.parametrize("F,want", [(900, 432904), (70, 4552), (772, 321928)])
def test_disc_fwd_workspace_and_prepared_floats(lib, F, want):
    assert lib.gic_disc_fwd_workspace_floats(F) == want
    assert lib.gic_disc_prepared_floats(F) == want


@pytest.mark.parametrize("shape,want,demb", zip(DISC_SHAPES, [44999184, 6000, 1074832], [29493904, 1056, 496400]))
def test_disc_bwd_workspace_floats_and_demb_offset(lib, shape, want, demb):
    N, L, De, R, F = shape
    assert lib.gic_disc_bwd_workspace_floats(*shape) == want
    assert lib.gic_disc_bwd_demb_offset_floats(*shape) == demb
    # demb[N*L*De] (read by the generator's factored backward) lies inside the workspace the caller allocated
    assert lib.gic_disc_bwd_demb_offset_floats(*shape) + N * L * De <= lib.gic_disc_bwd_workspace_floats(*shape)


@pytest.mark.parametrize("shape,want", [((256, 10000, 512), 26732100), ((128, 30000, 1024), 131733316), ((3, 37, 12), 3172)])
def test_decode_fwd_workspace_floats(lib, shape, want):
    assert lib.gic_decode_fwd_workspace_floats(*shape) == want


@pytest.mark.parametrize("shape,want", [((256, 20, 512, 512, 1), 21233664), ((3, 5, 12, 20, 2), 4320)])
def test_decode_saved_floats(lib, shape, want):
    assert lib.gic_decode_saved_floats(*shape) == want


@pytest.mark.parametrize("shape,want", [((256, 20, 10000, 512, 512, 1), 96920576), ((3, 5, 37, 12, 20, 2), 4756)])
def test_decode_bwd_workspace_floats(lib, shape, want):
    assert lib.gic_decode_bwd_workspace_floats(*shape) == want
