"""Coordinate transformations between the WGS 84 CRSs that need no datum shift.

Supported: EPSG:4326 (x = longitude, y = latitude in degrees, the axis order of the reference's
bboxes), EPSG:3857 (spherical Web Mercator on R = 6378137 m) and the WGS 84 UTM zones
EPSG:32601-32660 (north) / 32701-32760 (south), which are transverse Mercator evaluated with
Krueger's series to sixth order in n (Karney, "Transverse Mercator with an accuracy of a few
nanometers", J. Geodesy 85, 2011, eqs. 7-11, 35-36).  Every other pair raises
``NotImplementedError``: those need a datum transformation this build does not pin.

The device warp (csrc/gm_warp.cu) evaluates the same formulas; ``KINDS`` / ``parse`` give the
(kind, zone) pair it takes.  Longitudes are not wrapped into [-180, 180).
"""
import re

import numpy as np

GEOGRAPHIC, MERCATOR, UTM = 0, 1, 2

R_MERCATOR = 6378137.0
A = 6378137.0
F = 1 / 298.257223563
K0 = 0.9996
FALSE_EASTING = 500000.0
FALSE_NORTHING_SOUTH = 10000000.0

_N = F / (2 - F)
E2 = F * (2 - F)
E = np.sqrt(E2)
# rectifying radius and the Krueger coefficients (Karney 2011, eqs. 14, 35, 36)
A_RECT = A / (1 + _N) * (1 + _N ** 2 / 4 + _N ** 4 / 64 + _N ** 6 / 256)


def _series(rows):
    n = _N
    return np.array([sum(c * n ** (k + 1) for k, c in enumerate(row)) for row in rows])


ALPHA = _series([
    (1 / 2, -2 / 3, 5 / 16, 41 / 180, -127 / 288, 7891 / 37800),
    (0, 13 / 48, -3 / 5, 557 / 1440, 281 / 630, -1983433 / 1935360),
    (0, 0, 61 / 240, -103 / 140, 15061 / 26880, 167603 / 181440),
    (0, 0, 0, 49561 / 161280, -179 / 168, 6601661 / 7257600),
    (0, 0, 0, 0, 34729 / 80640, -3418889 / 1995840),
    (0, 0, 0, 0, 0, 212378941 / 319334400),
])
BETA = _series([
    (1 / 2, -2 / 3, 37 / 96, -1 / 360, -81 / 512, 96199 / 604800),
    (0, 1 / 48, 1 / 15, -437 / 1440, 46 / 105, -1118711 / 3870720),
    (0, 0, 17 / 480, -37 / 840, -209 / 4480, 5569 / 90720),
    (0, 0, 0, 4397 / 161280, -11 / 504, -830251 / 7257600),
    (0, 0, 0, 0, 4583 / 161280, -108847 / 3991680),
    (0, 0, 0, 0, 0, 20648693 / 638668800),
])


def parse(projection):
    """(kind, zone) of a projection string, or None when it is not one of the CRSs above.
    ``zone`` is 0 for EPSG:4326 / 3857, +z for UTM zone z north and -z for zone z south."""
    m = re.match(r"^EPSG:(\d+)$", str(projection).strip(), flags=re.IGNORECASE)
    if not m:
        return None
    code = int(m.group(1))
    if code == 4326:
        return GEOGRAPHIC, 0
    if code == 3857:
        return MERCATOR, 0
    if 32601 <= code <= 32660:
        return UTM, code - 32600
    if 32701 <= code <= 32760:
        return UTM, -(code - 32700)
    return None


def crs_pair(src, dst):
    """The parsed (src, dst) pair; NotImplementedError when either is unsupported."""
    a, b = parse(src), parse(dst)
    if a is None or b is None:
        raise NotImplementedError(
            "coordinate transformation {} -> {} needs a datum transformation (pyproj/GDAL), which "
            "this build does not use; supported are EPSG:4326, EPSG:3857 and the WGS 84 UTM "
            "zones".format(src, dst))
    return a, b


def is_separable(src, dst):
    """True when x maps to x and y to y independently (EPSG:4326 <-> EPSG:3857)."""
    return {src[0], dst[0]} == {GEOGRAPHIC, MERCATOR}


def central_meridian(zone):
    return 6.0 * abs(zone) - 183.0


# --- to / from geographic degrees -------------------------------------------------------------


def mercator_forward(lon, lat):
    """EPSG:3857 from degrees; |lat| = 90 gives +-inf, |lat| > 90 gives NaN."""
    lat = np.where(np.abs(lat) > 90, np.nan, lat)
    x = R_MERCATOR * np.radians(lon)
    with np.errstate(divide="ignore", invalid="ignore"):
        y = R_MERCATOR * np.arctanh(np.sin(np.radians(lat)))
    return x, y


def mercator_inverse(x, y):
    lon = np.degrees(x / R_MERCATOR)
    lat = np.degrees(2 * np.arctan(np.exp(y / R_MERCATOR)) - np.pi / 2)
    return lon, lat


def utm_forward(lon, lat, zone):
    """UTM easting / northing of ``zone`` (signed as in ``parse``) from degrees."""
    lat = np.where(np.abs(lat) > 90, np.nan, lat)
    phi = np.radians(lat)
    lam = np.radians(lon - central_meridian(zone))
    with np.errstate(divide="ignore", invalid="ignore"):
        s = np.sin(phi)
        # tangent of the conformal latitude (Karney 2011, eqs. 7-9)
        tau = np.tan(phi)
        sigma = np.sinh(E * np.arctanh(E * s))
        tau_c = tau * np.sqrt(1 + sigma ** 2) - sigma * np.sqrt(1 + tau ** 2)
        xi_c = np.arctan2(tau_c, np.cos(lam))
        eta_c = np.arcsinh(np.sin(lam) / np.hypot(tau_c, np.cos(lam)))
        z = xi_c + 1j * eta_c
        zeta = z + sum(ALPHA[j] * np.sin(2 * (j + 1) * z) for j in range(6))
    x = FALSE_EASTING + K0 * A_RECT * zeta.imag
    y = K0 * A_RECT * zeta.real + (FALSE_NORTHING_SOUTH if zone < 0 else 0.0)
    return x, y


def utm_inverse(x, y, zone):
    """Degrees from UTM easting / northing of ``zone``."""
    xi = (y - (FALSE_NORTHING_SOUTH if zone < 0 else 0.0)) / (K0 * A_RECT)
    eta = (x - FALSE_EASTING) / (K0 * A_RECT)
    z = xi + 1j * eta
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        zc = z - sum(BETA[j] * np.sin(2 * (j + 1) * z) for j in range(6))
        xi_c, eta_c = zc.real, zc.imag
        tau_c = np.sin(xi_c) / np.hypot(np.sinh(eta_c), np.cos(xi_c))
        lam = np.arctan2(np.sinh(eta_c), np.cos(xi_c))
        # conformal -> geographic latitude: Newton on tau (Karney 2011, eqs. 19-21)
        tau = tau_c.copy()
        for _ in range(3):
            sigma = np.sinh(E * np.arctanh(E * tau / np.sqrt(1 + tau ** 2)))
            tc = tau * np.sqrt(1 + sigma ** 2) - sigma * np.sqrt(1 + tau ** 2)
            dtau = ((tau_c - tc) / np.sqrt(1 + tc ** 2) * (1 + (1 - E2) * tau ** 2)
                    / ((1 - E2) * np.sqrt(1 + tau ** 2)))
            tau = tau + dtau
    lat = np.degrees(np.arctan(tau))
    lon = np.degrees(lam) + central_meridian(zone)
    return lon, lat


def _to_degrees(x, y, crs):
    kind, zone = crs
    if kind == GEOGRAPHIC:
        return x, y
    if kind == MERCATOR:
        return mercator_inverse(x, y)
    return utm_inverse(x, y, zone)


def _from_degrees(lon, lat, crs):
    kind, zone = crs
    if kind == GEOGRAPHIC:
        return lon, np.where(np.abs(lat) > 90, np.nan, lat)
    if kind == MERCATOR:
        return mercator_forward(lon, lat)
    return utm_forward(lon, lat, zone)


def transform_xy(x, y, src, dst):
    """(x, y) float64 arrays from parsed CRS ``src`` to ``dst`` (see ``parse``)."""
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    if src == dst:
        return x, y
    lon, lat = _to_degrees(x, y, src)
    return _from_degrees(lon, lat, dst)


def transform(xy, src, dst):
    """N x 2 float64 coordinates from projection ``src`` to ``dst`` (projection strings).
    Non-finite results mark points the target CRS cannot represent (e.g. a pole in EPSG:3857)."""
    a, b = crs_pair(src, dst)
    xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
    x, y = transform_xy(xy[:, 0], xy[:, 1], a, b)
    return np.stack([x, y], axis=1)
