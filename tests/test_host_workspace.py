"""Workspace sizes of the C ABI (no GPU): K6's workspace holds the scan scratch and the prefix-group index of up to nf
groups of four mask words; ordered compaction needs only its offsets, so a level's select does not pay for the index."""


def test_workspace_sizes():
    from ppopt_b200 import _lib
    lib = _lib.load()
    chunk = 2048   # csrc/k6_children.cu SCAN_CHUNK
    for n in (1, 2, 255, 256, 257, 2047, 2048, 2049, 100000, 3776565, 74554385):
        nb = (n + chunk - 1) // chunk
        sel, k6 = lib.ppgpu_select_workspace_bytes(n), lib.ppgpu_scan_workspace_bytes(n)
        # offsets (n + 1), block sums (+ total), one result slot
        assert sel == 8 * (n + 1 + nb + 3), n
        # block sums, header, table (>= 2 int32 slots per group and >= nf + 1 scan words), {start, E[4]} per group
        assert k6 >= 8 * (nb + 2 + 4 + max(2 * n + 2, 512) + 5 * n), n
        assert k6 >= sel
    assert lib.ppgpu_select_workspace_bytes(74554385) < 0.6e9 + 8 * 74554385
