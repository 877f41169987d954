"""Workspace queries of the Euclid filter (no GPU needed): from 9 references up it is sized for the tensor-core path (fp16 rows,
the reference bias, the candidates' scales and the re-check lists); up to 8 it stays the exact kernel's header."""


def test_euclid_workspace_bytes(ffr_lib):
    assert ffr_lib.ffr_filter_workspace_bytes(8, 1000, 128, 0, 1) == 256
    ws = ffr_lib.ffr_filter_workspace_bytes(9, 1000, 128, 0, 1)
    assert ws > 256
    assert ws >= 9 * 128 * 2 + 1000 * 128 * 2 + 256 * 4 + 1000 * 4 + 1000 * 16
    # fp16 rows are refused for Euclid: nothing beyond the header for them
    assert ffr_lib.ffr_filter_workspace_bytes(9, 1000, 128, 1, 1) == 256
    # dim > 512 keeps the exact kernel
    assert ffr_lib.ffr_filter_workspace_bytes(100, 1000, 640, 0, 1) == 256
