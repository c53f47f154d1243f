"""The WGS 84 coordinate transformations of crs.py pinned by closed forms and by properties
(no PROJ here): Web Mercator values, the UTM meridian arc against numerical quadrature,
forward / inverse round trips and conformality; and the geometry helpers built on them."""
import warnings

import numpy as np
import pytest
from scipy.integrate import IntegrationWarning, quad

from dask_geomodeling_b200 import crs, utils

PI_R = 20037508.342789244


def test_web_mercator_closed_form():
    xy = crs.transform([[180.0, 0.0], [0.0, 85.0511287798066], [-180.0, -85.0511287798066]],
                       "EPSG:4326", "EPSG:3857")
    np.testing.assert_allclose(xy, [[PI_R, 0.0], [0.0, PI_R], [-PI_R, -PI_R]], rtol=0, atol=1e-6)
    back = crs.transform(xy, "EPSG:3857", "EPSG:4326")
    np.testing.assert_allclose(back[1], [0.0, 85.0511287798066], atol=1e-11)
    poles = crs.transform([[0.0, 90.0], [0.0, -90.0], [0.0, 91.0]], "EPSG:4326", "EPSG:3857")
    assert poles[0, 1] == np.inf and poles[1, 1] == -np.inf and np.isnan(poles[2, 1])


def meridian_arc(lat):
    a, e2 = crs.A, crs.E2
    with warnings.catch_warnings():   # the requested tolerance is below what quad can certify
        warnings.simplefilter("ignore", IntegrationWarning)
        return quad(lambda p: a * (1 - e2) / (1 - e2 * np.sin(p) ** 2) ** 1.5, 0.0, np.radians(lat),
                    epsabs=1e-10, epsrel=1e-14, limit=200)[0]


@pytest.mark.parametrize("zone", [1, 31, 60])
def test_utm_central_meridian_is_the_scaled_meridian_arc(zone):
    lats = np.linspace(0.0, 84.0, 43)
    lon = np.full_like(lats, crs.central_meridian(zone))
    north = crs.transform(np.stack([lon, lats], 1), "EPSG:4326", "EPSG:{}".format(32600 + zone))
    assert (north[:, 0] == 500000.0).all()
    expected = np.array([0.9996 * meridian_arc(lat) for lat in lats])
    assert np.abs(north[:, 1] - expected).max() < 1e-3
    south = crs.transform(np.stack([lon, -lats], 1), "EPSG:4326", "EPSG:{}".format(32700 + zone))
    np.testing.assert_allclose(south[:, 1], 10000000.0 - expected, rtol=0, atol=1e-3)


@pytest.mark.parametrize("code", [32601, 32631, 32660, 32701, 32733, 32760])
def test_utm_round_trip(code):
    zone = code - 32600 if code < 32700 else code - 32700
    rng = np.random.default_rng(code)
    lon = crs.central_meridian(zone) + rng.uniform(-3.0, 3.0, 2000)
    lat = rng.uniform(0.0, 84.0, 2000) if code < 32700 else rng.uniform(-80.0, 0.0, 2000)
    lonlat = np.stack([lon, lat], 1)
    xy = crs.transform(lonlat, "EPSG:4326", "EPSG:{}".format(code))
    back = crs.transform(xy, "EPSG:{}".format(code), "EPSG:4326")
    assert np.abs(back - lonlat).max() < 1e-11
    again = crs.transform(back, "EPSG:4326", "EPSG:{}".format(code))
    assert np.abs(again - xy).max() < 1e-6


def jacobian(lon, lat, projection, h=1e-3):
    """Derivatives of (x, y) per metre east and per metre north on the ellipsoid (fourth-order
    central differences of step h degrees)."""
    def d(dlon, dlat):
        f = lambda k: crs.transform([[lon + k * dlon, lat + k * dlat]], "EPSG:4326", projection)[0]
        return (-f(2) + 8 * f(1) - 8 * f(-1) + f(-2)) / 12

    a, e2 = crs.A, crs.E2
    phi = np.radians(lat)
    w = np.sqrt(1 - e2 * np.sin(phi) ** 2)
    east = a * np.cos(phi) / w * np.radians(h)          # metres per h degrees of longitude
    north = a * (1 - e2) / w ** 3 * np.radians(h)       # metres per h degrees of latitude
    return d(h, 0) / east, d(0, h) / north


@pytest.mark.parametrize("lon,lat", [(3.0, 10.0), (1.0, 45.0), (5.5, 60.0), (0.5, 75.0), (4.0, -30.0)])
def test_utm_is_conformal(lon, lat):
    projection = "EPSG:32631" if lat >= 0 else "EPSG:32731"
    d_east, d_north = jacobian(lon, lat, projection)
    k_east, k_north = np.hypot(*d_east), np.hypot(*d_north)
    assert abs(k_east - k_north) / k_east < 1e-9
    assert abs(np.dot(d_east, d_north)) / (k_east * k_north) < 1e-9
    if lon == 3.0:
        assert abs(k_east - 0.9996) < 1e-9


def test_geometry_helpers_agree():
    shell = [(4.0, 50.0), (6.0, 50.5), (5.5, 52.0), (4.2, 51.5)]
    hole = [(4.8, 50.8), (5.2, 50.8), (5.0, 51.2)]
    polygon = utils.Polygon(shell, [hole])
    for dst in ("EPSG:3857", "EPSG:32631", "EPSG:32733"):
        moved = utils.shapely_transform(polygon, "EPSG:4326", dst)
        soup = utils.PolygonSoup([polygon]).transformed("EPSG:4326", dst)
        np.testing.assert_array_equal(soup.xy, np.concatenate([moved.exterior.coords, moved.interiors[0].coords]))
        assert tuple(soup.bounds()[0]) == moved.bounds
        extent = utils.Extent(polygon.bounds, "EPSG:4326").transformed(dst)
        x1, y1, x2, y2 = polygon.bounds
        corners = crs.transform([(x1, y1), (x1, y2), (x2, y1), (x2, y2)], "EPSG:4326", dst)
        assert extent.projection == dst
        assert extent.bbox == (corners[:, 0].min(), corners[:, 1].min(), corners[:, 0].max(), corners[:, 1].max())
        multi = utils.shapely_transform(utils.MultiPolygon([polygon, utils.box(7, 50, 8, 51)]), "EPSG:4326", dst)
        np.testing.assert_array_equal(multi.geoms[0].exterior.coords, moved.exterior.coords)
        point = utils.shapely_transform(utils.Point(5.0, 51.0), "EPSG:4326", dst)
        assert (point.x, point.y) == tuple(crs.transform([(5.0, 51.0)], "EPSG:4326", dst)[0])
    assert utils.Extent((1, 2, 3, 4), "EPSG:3857").transformed("epsg:3857").bbox == (1, 2, 3, 4)


@pytest.mark.parametrize("pair", [("EPSG:28992", "EPSG:4326"), ("EPSG:4326", "EPSG:28992"),
                                  ("EPSG:4258", "EPSG:3857"), ("EPSG:25831", "EPSG:32631"),
                                  ('GEOGCS["WGS 84"]', "EPSG:4326")])
def test_other_crs_pairs_still_raise(pair):
    src, dst = pair
    with pytest.raises(NotImplementedError):
        utils.Extent((0, 0, 1, 1), src).transformed(dst)
    with pytest.raises(NotImplementedError):
        utils.shapely_transform(utils.box(0, 0, 1, 1), src, dst)
    with pytest.raises(NotImplementedError):
        utils.PolygonSoup([utils.box(0, 0, 1, 1)]).transformed(src, dst)
    with pytest.raises(NotImplementedError):
        crs.transform([[0.0, 0.0]], src, dst)


def test_parse():
    assert crs.parse("epsg:4326") == (crs.GEOGRAPHIC, 0) and crs.parse("EPSG:3857") == (crs.MERCATOR, 0)
    assert crs.parse("EPSG:32631") == (crs.UTM, 31) and crs.parse("EPSG:32733") == (crs.UTM, -33)
    assert crs.parse("EPSG:32661") is None and crs.parse("EPSG:32700") is None and crs.parse("EPSG:28992") is None
