"""Host I/O around the path (SURVEY.md §8f row 1) and the kept CLI surface (run_real_data_script.py:18-62,82-93)."""
import gzip
import os
import struct

import numpy as np
import pytest

import run_real_data_script as cli
import run_real_data_script_ROI_based_estimation as cli_roi
from multicomponent_t2_toolbox_b200 import nifti_io


def test_nifti_roundtrip_gz_and_plain(tmp_path):
    rng = np.random.default_rng(0)
    a = rng.uniform(size=(5, 4, 3, 6))
    aff = np.array([[2.0, 0, 0, -10], [0, 2.5, 0, 5], [0, 0, 3.0, 1], [0, 0, 0, 1]])
    for name in ("x.nii.gz", "y.nii"):
        p = str(tmp_path / name)
        nifti_io.save(a, p, affine=aff)
        im = nifti_io.load(p)
        assert im.shape == a.shape
        assert np.array_equal(im.get_fdata(), a) and np.allclose(im.affine, aff)
    raw = gzip.open(str(tmp_path / "x.nii.gz")).read()
    assert struct.unpack("<i", raw[:4])[0] == 348 and raw[344:347] == b"n+1"
    assert struct.unpack("<h", raw[70:72])[0] == 64            # float64, like the reference's outputs
    assert len(raw) == 352 + a.size * 8
    assert raw[352:360] == struct.pack("<d", a[0, 0, 0, 0])      # Fortran order: x runs fastest
    assert raw[360:368] == struct.pack("<d", a[1, 0, 0, 0])


def test_nifti_int_mask_and_scaling(tmp_path):
    m = (np.arange(24).reshape(2, 3, 4) % 2).astype(np.int16)
    p = str(tmp_path / "m.nii.gz")
    nifti_io.save(m, p)
    im = nifti_io.load(p)
    assert np.array_equal(im.get_fdata(), m.astype(float))
    im.header["scl_slope"], im.header["scl_inter"] = 2.0, 1.0
    assert np.array_equal(im.get_fdata(), 2.0 * m + 1.0)
    with pytest.raises(ValueError):
        (tmp_path / "bad.nii").write_bytes(b"\x00" * 400)
        nifti_io.load(str(tmp_path / "bad.nii"))


def test_parallel_gzip_is_one_standard_member(tmp_path):
    """The threaded deflate (nifti_io._gzip_pieces) must give an ordinary gzip file: ONE member (a reader that stops
    after the first member sees everything), correct CRC/size trailer, same bytes for any thread count, chunk
    boundaries (4 MiB) crossed, empty payload handled."""
    import zlib
    rng = np.random.default_rng(1)
    a = rng.integers(0, 4, size=(96, 96, 30, 6)).astype(np.float64)     # 13.3 MB -> four deflate chunks
    files = []
    for th in (1, 3, 8):
        p = str(tmp_path / ("t%d.nii.gz" % th))
        nifti_io.save(a, p, threads=th)
        files.append(open(p, "rb").read())
    assert files[0] == files[1] == files[2]
    blob = files[0]
    d = zlib.decompressobj(31)                                         # one member only
    raw = d.decompress(blob)
    assert d.eof and d.unused_data == b"" and len(raw) == 352 + a.nbytes
    assert struct.unpack("<II", blob[-8:]) == (zlib.crc32(raw), len(raw) & 0xFFFFFFFF)
    assert np.array_equal(nifti_io.load(str(tmp_path / "t8.nii.gz")).get_fdata(), a)
    assert b"".join(nifti_io._gzip_pieces(b"", 1, 4)) and gzip.decompress(b"".join(nifti_io._gzip_pieces(b"", 1, 4))) == b""
    for n in (1, nifti_io._GZ_CHUNK - 1, nifti_io._GZ_CHUNK, nifti_io._GZ_CHUNK + 1):
        buf = rng.integers(0, 3, size=n, dtype=np.uint8).tobytes()
        assert gzip.decompress(b"".join(nifti_io._gzip_pieces(buf, 1, 4))) == buf


def test_nifti_big_endian_qform_and_shapes(tmp_path):
    """A big-endian file with the affine in the qform (what some scanners write) reads like nibabel reads it; arrays of
    every rank the toolbox writes (3-D maps, 4-D spectra, a singleton last axis) round-trip."""
    a = np.arange(2 * 3 * 4, dtype=np.float32).reshape(2, 3, 4)
    hdr = bytearray(348)
    struct.pack_into(">i", hdr, 0, 348)
    struct.pack_into(">8h", hdr, 40, 3, 2, 3, 4, 1, 1, 1, 1)
    struct.pack_into(">hh", hdr, 70, 16, 32)
    struct.pack_into(">8f", hdr, 76, -1.0, 2.0, 3.0, 4.0, 1.0, 1.0, 1.0, 1.0)
    struct.pack_into(">3f", hdr, 108, 352.0, 0.0, 0.0)
    struct.pack_into(">hh", hdr, 252, 1, 0)
    struct.pack_into(">6f", hdr, 256, 0.0, 0.0, 0.0, 7.0, 8.0, 9.0)
    hdr[344:348] = b"n+1\x00"
    p = str(tmp_path / "be.nii")
    open(p, "wb").write(bytes(hdr) + b"\x00" * 4 + a.astype(">f4").tobytes(order="F"))
    im = nifti_io.load(p)
    assert np.array_equal(im.get_fdata(), a.astype(np.float64))
    assert np.allclose(im.affine, [[2, 0, 0, 7], [0, 3, 0, 8], [0, 0, -4, 9], [0, 0, 0, 1]])   # qfac = -1 flips z
    rng = np.random.default_rng(2)
    for shape in ((4, 5, 6), (4, 5, 6, 1), (3, 2, 2, 7), (6,)):
        x = rng.uniform(size=shape)
        q = str(tmp_path / "s.nii.gz")
        nifti_io.save(x, q)
        assert np.array_equal(nifti_io.load(q).get_fdata(), x)


@pytest.mark.parametrize("script,mod", [("run_real_data_script.py", "cli"),
                                        ("run_real_data_script_ROI_based_estimation.py", "cli_roi")])
def test_cli_flag_table_equals_reference_argparse(script, mod):
    """Flag / type / default / choices / required of every option, diffed against the reference's own argparse block
    (run_real_data_script.py:18-62, run_real_data_script_ROI_based_estimation.py:18-52) as recorded in
    tests/golden/reference_cli_flags.json."""
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_cli_flags.json")) as fh:
        ref = json.load(fh)[script]
    ours = {f: dict(type=t.__name__, default=d, choices=c, required=r)
            for f, t, d, c, r, _ in globals()[mod]._FLAGS}
    assert ours == ref


def test_cli_flags_match_reference():
    argv = ("--path_to_folder /data/ --input Data.nii.gz --mask Mask.nii.gz --minTE 10.68 --nTE 32 --TR 1000 "
            "--FA_method spline --FA_smooth yes --denoise None --reg_method X2 --reg_matrix I "
            "--myelin_T2=40 --savefig no --savefig_slice 30").split()   # --myelin_T2 relies on prefix matching
    a = cli.build_parser().parse_args(argv)
    assert a.myelin_T2_cutoff == 40.0 and a.reg_method == "X2" and a.FA_method == "spline" and a.nTE == 32
    assert a.numcores == -1                                           # optional, default -1 (= all), like the reference
    assert cli.build_parser().parse_args(argv + ["--numcores", "2"]).numcores == 2
    with pytest.raises(SystemExit):
        cli.build_parser().parse_args(argv[:-2])                  # every other flag is required, like the reference
    with pytest.raises(SystemExit):
        cli.build_parser().parse_args([x if x != "X2" else "Tikhonov" for x in argv])