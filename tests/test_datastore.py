"""Project input side (SURVEY.md 8(f) rank 3): OMEGA .ini parser against the reference's readini
(golden fixture), SEG-Y reader against the format definition, the DFT pair, and the datastores."""
import json
import pickle

import numpy as np
import pytest

from zephyr_b200 import datastore as zds


def jsonable(d):
    return {k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in d.items()}


def test_readini_matches_reference(golden, tmp_path):
    g = golden('ini')
    fn = tmp_path / 'proj.ini'
    fn.write_text(g['text'].item())
    mine = zds.readini(str(fn))
    assert json.dumps(jsonable(mine), sort_keys=True) == g['parsed'].item()
    assert isinstance(mine['freqs'], np.ndarray) and mine['srcs'].shape == (6, 3) and mine['recs'].shape == (9, 3)
    # writer/reader round trip
    again = zds.readini(zds.writeini(str(tmp_path / 'again.ini'), mine))
    assert json.dumps(jsonable(again), sort_keys=True) == g['parsed'].item()


def test_ibm_floats_and_segy_roundtrip(tmp_path):
    words = np.array([0xC276A000, 0x42640000, 0x00000000, 0x41100000, 0x40800000, 0xBF100000], dtype=np.uint32)
    assert np.array_equal(zds.ibm2ieee(words), [-118.625, 100.0, 0.0, 1.0, 0.5, -1.0 / 256.0])
    rng = np.random.default_rng(0)
    tr = np.concatenate([rng.uniform(1500., 4500., size=(7, 33)), rng.normal(size=(2, 33)) * 1e-3, np.zeros((1, 33))])
    tr[0, :4] = [1.0, 16.0, 256.0, 1.0 / 16.0]                                      # exact powers of 16
    for fmt, endian, tol in ((1, 'big', 2.0 ** -20), (5, 'big', 0.), (5, 'little', 0.), (1, 'little', 2.0 ** -20)):
        fn = zds.write_segy(str(tmp_path / ('m%d%s.segy' % (fmt, endian))), tr, fmt=fmt, endian=endian)
        sf = zds.SEGYFile(fn)
        assert sf.endian == endian and sf.format == fmt and sf.shape == (10, 33) and len(sf) == 10
        got = sf[:]
        assert got.dtype == np.float32
        want = tr.astype(np.float32)
        assert np.all(np.abs(got - want) <= tol * np.abs(want) + (0 if tol == 0 else 1e-45))
        assert np.array_equal(sf[2], got[2]) and np.array_equal(sf[1:8:3], got[1:8:3])
        assert sf.trace_header(4, 0, size=4) == 5 and sf.trace_header(4, 114, signed=False) == 33
    with pytest.raises(ValueError):
        (tmp_path / 'short.segy').write_bytes(b'\0' * 100)
        zds.SEGYFile(str(tmp_path / 'short.segy'))


def test_source_terms_dft_convention():
    """.src time series -> per-frequency source terms: e^{+i...}/N convention (time.py:47-49), zero frequency dropped."""
    rng = np.random.default_rng(1)
    x = rng.normal(size=(3, 8))
    st = zds.source_terms(x, 4)
    assert st.shape == (4, 3)
    assert np.allclose(st.T, (np.conj(np.fft.fft(x, axis=1)) / 8)[:, 1:5])
    assert zds.source_terms(x[0], 4).shape == (4, 1)
    with pytest.raises(AssertionError):
        zds.source_terms(x[:, :7], 4)


def make_project(tmp_path, name='proj', nx=24, nz=30, nsrc=3, with_src=True, nfreq=3):
    rng = np.random.default_rng(3)
    freqs = 4. * np.arange(1, nfreq + 1)
    vp = 2000. + 1000. * rng.uniform(size=(nx, nz))                                  # traces along x
    qp = 1. / (50. + 100. * rng.uniform(size=(nx, nz)))
    srcs = np.column_stack([np.linspace(40., (nx - 5) * 10., nsrc), np.full(nsrc, 50.), np.ones(nsrc)])
    recs = np.column_stack([np.linspace(20., (nx - 3) * 10., 8), np.full(8, 60.), np.ones(8)])
    settings = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'freqs': freqs, 'freqbase': 4., 'srcs': srcs, 'recs': recs,
                'isreg': 4, 'tau': 999.999, 'fst': True}
    base = str(tmp_path / name)
    zds.writeini(base + '.ini', settings)
    zds.write_segy(base + '.vp', vp)
    zds.write_segy(base + '.qp', qp, fmt=5)
    wav = None
    if with_src:
        wav = rng.normal(size=(1, 2 * len(freqs)))
        zds.write_segy(base + '.src', wav, fmt=5)
    (tmp_path / (name + '.notes')).write_text('not a project file')
    return base, settings, vp, qp, wav


def test_fullwv_datastore(tmp_path):
    base, settings, vp, qp, wav = make_project(tmp_path)
    ds = zds.FullwvDatastore(base)
    assert sorted(ds.keys()) == ['proj.qp', 'proj.src', 'proj.vp'] and '.vp' in ds and '.rho' not in ds
    assert 'comprising 3 files' in repr(ds)
    assert ds['.vp'].shape == (24, 30) and ds['.vp', 2].shape == (30,) and ds['proj.vp', 1:3].shape == (2, 30)
    with pytest.raises(KeyError):
        ds['.rho']
    sc = ds.systemConfig
    assert (sc['nx'], sc['nz'], sc['dx'], sc['ireg'], sc['freqBase']) == (24, 30, 10., 4, 4.)
    assert sc['tau'] == np.inf and sc['freeSurf'] == (True, False, False, False)
    assert sc['c'].shape == (30, 24) and np.allclose(sc['c'], vp.T, rtol=2e-6)
    assert np.allclose(sc['Q'], 1. / qp.T.astype(np.float32), rtol=1e-6)
    assert np.array_equal(sc['geom']['src'], settings['srcs'][:, :2]) and sc['geom']['mode'] == 'fixed'
    assert sc['geom']['rec'].shape == (8, 2) and list(sc['freqs']) == [4., 8., 12.]
    st = sc['sterms']
    assert st.shape == (3, 1)
    w32 = wav.astype(np.float32).astype(np.float64)
    assert np.allclose(st[:, 0], (np.conj(np.fft.fft(w32[0])) / 6)[1:4])
    with pytest.raises(Exception):
        zds.FullwvDatastore(str(tmp_path / 'nothere'))
    # data spooling: interleaved re/im traces per frequency (db.py:254-266)
    rng = np.random.default_rng(4)
    d = rng.normal(size=(3, 8)) + 1j * rng.normal(size=(3, 8))                        # (nsrc, nrec)
    il = np.empty((6, 8))
    il[::2], il[1::2] = d.real, d.imag
    zds.write_segy(base + '.utobs8.000', il, fmt=5)
    ds = zds.FullwvDatastore(base)
    got = list(ds.spoolData(fid=slice(1, 2)))
    assert len(got) == 1 and np.allclose(got[0], d.T, rtol=1e-6)
    with pytest.raises(ValueError):
        list(ds.spoolData())
    # 2.5-D geometry columns x, y, z, w
    settings25 = dict(settings, srcs=np.column_stack([settings['srcs'][:, 0], 0 * settings['srcs'][:, 0], settings['srcs'][:, 1:]]),
                      recs=np.column_stack([settings['recs'][:, 0], 0 * settings['recs'][:, 0], settings['recs'][:, 1:]]))
    zds.writeini(str(tmp_path / 'p25.ini'), settings25)
    sc25 = zds.FullwvDatastore(str(tmp_path / 'p25')).systemConfig
    assert np.array_equal(sc25['geom']['src'], settings['srcs'][:, :2]) and 'c' not in sc25


def test_flat_and_pickle_datastores(tmp_path):
    (tmp_path / 'flat.py').write_text("import numpy as np\nsystemConfig = {'nx': 5, 'nz': 6, 'c': 2500. * np.ones((6, 5))}\n")
    sc = zds.FlatDatastore(str(tmp_path / 'flat')).systemConfig
    assert sc['nx'] == 5 and sc['c'].shape == (6, 5)
    with open(tmp_path / 'pick.pickle', 'wb') as fp:
        pickle.dump({'nx': 7, 'freqs': [1., 2.]}, fp)
    assert zds.PickleDatastore(str(tmp_path / 'pick')).systemConfig == {'nx': 7, 'freqs': [1., 2.]}
