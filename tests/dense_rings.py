"""Dense-ring sweeps and a host-side mirror of the extraction kernels' path choice (lvo_extract.cuh).

The standard synthetic sweeps have at most 1875 points per ring, so they only reach the fast extraction path with
k_lessflat_voxel<128>.  The fixtures here are the same scene cast with more azimuth columns (lvo_synth_sweep_res), some with
one ring cut to a chosen length, so that every reachable branch of k_sector_sort / k_lessflat_voxel<256> / k_sector_pick runs:

  ring of n points:  E - S = n - 11 (scanStartInd = start + 5, scanEndInd = end - 6), RL = E - S + 12, mmax = (E - S + 5) / 6 + 1
  fast path          RL <= 4096 and mmax <= 512, i.e. E - S <= 3066; less-flat candidates (label <= 0 in [S, E - 1]) <= 2048 take
                     k_lessflat_voxel<128>, more take <256>
  generic kernel     every other ring with E - S >= 6: picked flags in shared memory when RL <= 4096, else in global memory; each
                     sector sort in shared memory when next_pow2(m) <= 3072, else in the lane's sort_scratch; the less-flat voxel sort
                     in shared memory when next_pow2(candidates) <= 3072, else in sort_scratch.
"""
import numpy as np

VLP16 = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
HDL64 = dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8)
PICK_RING_SMEM, PICK_SMEM_KEYS = 4096, 3072   # LVO_PICK_RING_SMEM, LVO_PICK_SMEM_KEYS

# name -> (model, seq, frame, naz, {ring: points kept}, thin), thin = (first ring, ring step, point step): keep every point step-th
# point of those rings.  The ring cuts of "boundaries" sit on both sides of every size limit of the kernels:
#   ring 0: 12299 points, E - S 12288, six sectors of 2048   ring 1: 12300 points, one sector of 2049 (sorted in sort_scratch)
#   ring 2: 4095 points, RL 4096                              ring 3: 4096 points, RL 4097 (picked flags in global memory)
#   ring 4: 3077 points, mmax 512 (fast path)                 ring 5: 3078 points, mmax 513 (generic kernel)
#   ring 6: 2090 points, 2048 less-flat candidates (<128>)    ring 7: 2111 points, 2049 candidates (<256>)
FIXTURES = {
    "vlp16_naz2700": (16, 0, 0, 2700, {}, None),
    "vlp16_naz3600": (16, 0, 0, 3600, {}, None),
    "vlp16_naz7200": (16, 0, 0, 7200, {}, None),
    "vlp16_naz20000": (16, 0, 0, 20000, {}, None),
    "hdl64_naz3000": (64, 0, 0, 3000, {}, None),
    "boundaries": (16, 0, 0, 13000, {0: 12299, 1: 12300, 2: 4095, 3: 4096, 4: 3077, 5: 3078, 6: 2090, 7: 2111}, None),
    # fast and generic rings in one lane (they share sort_scratch: the fast path keeps its keys at sp, the generic kernel at 2 sp)
    "mixed": (16, 1, 2, 7200, {}, (1, 2, 3)),
}
# paths each fixture must reach (a ring reaches the union of its tags; "ring k: tags" must hold for that ring)
EXPECT = {
    "vlp16_naz2700": ({"fast", "lfv256"}, {}),
    "vlp16_naz3600": ({"generic", "flags_smem", "sort_smem", "lf_global"}, {}),
    "vlp16_naz7200": ({"generic", "flags_global", "sort_smem", "lf_global"}, {}),
    "vlp16_naz20000": ({"generic", "flags_global", "sort_global"}, {}),
    "hdl64_naz3000": ({"fast", "lfv256"}, {}),
    "boundaries": (set(), {0: {"generic", "flags_global", "sort_smem"}, 1: {"generic", "flags_global", "sort_smem", "sort_global"},
                           2: {"generic", "flags_smem"}, 3: {"generic", "flags_global"}, 4: {"fast"}, 5: {"generic", "flags_smem"},
                           6: {"fast", "lfv128"}, 7: {"fast", "lfv256"}}),
    "mixed": ({"fast", "lfv256", "generic", "flags_global"}, {}),
}


def vlp16_ring(pts):
    """Beam index of each point of a VLP-16 sweep (elevations -15..15 deg, 2 deg apart: rounding is exact)."""
    el = np.degrees(np.arctan2(pts[:, 2].astype(np.float64), np.hypot(pts[:, 0], pts[:, 1])))
    return np.rint((el + 15.0) / 2.0).astype(np.int64)


def make(synth, name):
    """(points, model, sensor settings) of one fixture."""
    model, seq, frame, naz, cut, thin = FIXTURES[name]
    pts, _ = synth.sweep(model, seq, frame, naz=naz)
    if cut or thin:
        assert model == 16
        ring = vlp16_ring(pts)
        keep = np.ones(len(pts), bool)
        for r, n in cut.items():
            keep[np.nonzero(ring == r)[0][n:]] = False
        if thin:
            r0, rstep, pstep = thin
            for r in range(r0, model, rstep):
                idx = np.nonzero(ring == r)[0]
                keep[np.setdiff1d(idx, idx[::pstep])] = False
        pts = np.ascontiguousarray(pts[keep])
    return pts, model, dict(VLP16 if model == 16 else HDL64)


def next_pow2(n):
    return 1 << max(0, int(n) - 1).bit_length()


def ring_paths(ref):
    """Per ring of an oracle extraction: (E - S, less-flat candidates, set of kernel paths the ring takes on the GPU)."""
    out = []
    for S, E in zip(ref["scan_start"], ref["scan_end"]):
        d = int(E) - int(S)
        if d < 6:
            out.append((d, 0, {"none"}))
            continue
        ncand = int((ref["label"][S:E] <= 0).sum())
        RL, mmax = d + 12, (d + 5) // 6 + 1
        tags = set()
        if RL <= PICK_RING_SMEM and mmax <= 512:
            tags.add("fast")
            if ncand:
                tags.add("lfv128" if ncand <= 2048 else "lfv256")
        else:
            tags |= {"generic", "flags_smem" if RL <= PICK_RING_SMEM else "flags_global"}
            if 6 * next_pow2(mmax) <= PICK_SMEM_KEYS:
                tags.add("joint")
            for j in range(6):
                m = (S + d * (j + 1) // 6 - 1) - (S + d * j // 6) + 1
                tags.add("sort_smem" if next_pow2(m) <= PICK_SMEM_KEYS else "sort_global")
            if ncand:
                tags.add("lf_smem" if next_pow2(ncand) <= PICK_SMEM_KEYS else "lf_global")
        out.append((d, ncand, tags))
    return out
