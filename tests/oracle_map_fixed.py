"""Localisation in a fixed map on the CPU oracle: process() (laserMapping.cpp:307-848) with the insertion (:737-783) and the per-cube
re-filter (:788-801) skipped.  The reference has no such mode; this is the definition lvo_set_lane_map_update(ctx, lane, 0) implements.

The oracle restatement (oracle/laser_mapping.hpp) is used as it is.  Insertion and re-filter come after everything a frame reports
(the pose, transformUpdate, the registered cloud), so skipping them changes only the map a frame leaves behind: the map before the
frame with the frame's cube-window shift (:312-507) applied.  A frame is therefore run in full and the map is then put back: the map
exported before the frame, each cube moved by the shift, the cubes that left the 21 x 21 x 11 window dropped.  TEST INFRASTRUCTURE."""
import numpy as np

from oracle_py import Oracle

W, H, D = 21, 21, 11


def shift_cubes(pts, cube, d):
    """The cube-window shift of :312-507 on an exported map: cube (i, j, k) moves to (i + d0, j + d1, k + d2); cubes that leave the
    window are dropped (the reference clears the recycled cube).  Points keep their order inside a cube."""
    i, j, k = cube % W + d[0], (cube // W) % H + d[1], cube // (W * H) + d[2]
    keep = (i >= 0) & (i < W) & (j >= 0) & (j < H) & (k >= 0) & (k < D)
    return pts[keep], (i + W * j + W * H * k)[keep].astype(np.int32)


class MapFixedOracle(Oracle):
    """Oracle with a map-update switch (on by default), honoured by mapping() and step()."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.map_update = True

    def set_map_update(self, on):
        self.map_update = bool(on)

    def cen(self):
        """laserCloudCen{Width,Height,Depth} as they are now."""
        return self._get(self.lib.lvo_oracle_mapping_log, (0, 5), np.int32)[3:6].copy()

    def _before(self):
        if self.map_update:
            return None
        return self.cen(), self.map_export(0), self.map_export(1)

    def _after(self, saved, mapped=True):
        if saved is None or not mapped:
            return
        cen0, (pc, cc), (ps, cs) = saved
        d = self.cen() - cen0
        for which, (p, c) in enumerate(((pc, cc), (ps, cs))):
            self.map_import(which, *shift_cubes(p, c, d))

    def mapping(self, *args, **kw):
        saved = self._before()
        r = super().mapping(*args, **kw)
        self._after(saved)
        return r

    def step(self, *args, **kw):
        saved = self._before()
        r = super().step(*args, **kw)
        self._after(saved, self.last_frame_mapped())
        return r
