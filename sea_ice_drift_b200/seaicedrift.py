"""``SeaIceDrift`` façade with the reference's interface (reference
sea_ice_drift/seaicedrift.py:23-88).  Pattern matching runs on the GPU; opening
Sentinel-1 files (Nansat/GDAL) and ORB feature tracking stay on the reference
path and are delegated to the ``sea_ice_drift`` package when it is installed;
``get_drift_coarse`` gives first-guess matches without it, on the GPU."""
from .pmlib import coarse_tracking, pattern_matching


class SeaIceDrift(object):
    def __init__(self, filename1, filename2, **kwargs):
        """``filename1/2``: Sentinel-1 file names (needs the reference package and
        Nansat), or two already opened Nansat-like objects (``n[1]``, ``shape()``,
        ``transform_points()``, ``get_corners()``)."""
        self.filename1, self.filename2 = filename1, filename2
        if isinstance(filename1, str):
            try:
                from sea_ice_drift.lib import get_n
            except ImportError as e:
                raise ImportError("opening files needs the reference package 'sea_ice_drift' (Nansat/GDAL); "
                                  "pass Nansat-like objects instead") from e
            self.n1, self.n2 = get_n(filename1, **kwargs), get_n(filename2, **kwargs)
        else:
            self.n1, self.n2 = filename1, filename2

    def get_drift_FT(self, **kwargs):
        """Feature tracking is out of this package's scope: delegated to the reference."""
        try:
            from sea_ice_drift.ftlib import feature_tracking
            from sea_ice_drift.lib import get_drift_vectors
        except ImportError as e:
            raise ImportError("get_drift_FT needs the reference package 'sea_ice_drift' (ORB feature tracking "
                              "stays on the reference path)") from e
        x1, y1, x2, y2 = feature_tracking(self.n1, self.n2, **kwargs)
        return get_drift_vectors(self.n1, x1, y1, self.n2, x2, y2, **kwargs)

    def get_drift_coarse(self, **kwargs):
        """Extension: the contract of get_drift_FT, ``(lon1, lat1, lon2, lat2)`` of matches on image 1 and image 2, from
        pattern matching on a box-downsampled copy of the pair (:func:`pmlib.coarse_tracking`, keywords there) instead
        of ORB feature tracking, so it needs neither the reference package nor host image processing."""
        x1, y1, x2, y2 = coarse_tracking(self.n1, self.n2, **kwargs)
        lon1, lat1 = self.n1.transform_points(x1, y1)
        lon2, lat2 = self.n2.transform_points(x2, y2)
        return lon1, lat1, lon2, lat2

    def get_drift_PM(self, lons, lats, lon1, lat1, lon2, lat2, **kwargs):
        """Same contract as the reference's get_drift_PM (seaicedrift.py:62-88):
        returns ``u, v, a, r, h, lon2_dst, lat2_dst`` shaped like ``lons``."""
        x1, y1 = self.n1.transform_points(lon1, lat1, 1)
        x2, y2 = self.n2.transform_points(lon2, lat2, 1)
        return pattern_matching(lons, lats, self.n1, x1, y1, self.n2, x2, y2, **kwargs)
