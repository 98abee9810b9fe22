"""The data formats either side of the path (SURVEY 8f #3, #4): the L9 CSV reader (src/main.c:77-128)
and the 25-column CSV row writer (src/main.c:243,320-352).  Host code of the C-ABI library, so these
run without a GPU.  Checkers: the reference's own readers (oracle/_ref where built, else their stored
answers, oracle_lib.check_ref), the oracle's
fscanf / snprintf restatements, and Python's correctly rounded '%.2f'."""
import importlib
import os

import numpy as np
import pytest

from oracle_lib import Oracle, RefLib, check_ref, ref_available

nav = importlib.import_module("nav-slam_b200")
synth = importlib.import_module("nav-slam_b200.synth")


@pytest.fixture(scope="module")
def oracle():
    return Oracle()


def _special_doubles(rng, n):
    """Magnitudes from denormal to 1e300, exact .xx5 ties, values that round across a power of ten."""
    v = [0.0, -0.0, 0.005, 0.015, 0.025, 0.125, 0.375, -0.125, 2.675, 1.005, 0.994999999999, 0.995, 9.995, 99.995,
         999.995, -999.995, 5e-324, -5e-324, 1e-3, 4.9999999e-3, 5.0000001e-3, 1e15, 123456789012345.67,
         2.0 ** 52 + 0.5, 2.0 ** 53, 2.0 ** 57, 2.0 ** 60, 1e22, 1e300, -1e300, 1.7976931348623157e308,
         float("inf"), float("-inf"), 1 / 3, -2 / 3, 1234.5, 0.5, 1.5, 2.5]
    k = rng.integers(0, 2 ** 20, n // 4)
    v += list(k / 8.0 + 0.005)                       # many land next to a tie
    v += list((k * 2 + 1) / 8.0)                     # x.125 / x.375 / x.625 / x.875: exact ties
    v += list(rng.standard_normal(n // 4) * 10.0 ** rng.integers(-8, 16, n // 4))
    v += list(np.ldexp(rng.random(n // 4) + 0.5, rng.integers(-1074, 1023, n // 4)) * rng.choice([-1, 1], n // 4))
    return np.array(v, dtype=np.float64)


def test_fixed2_matches_printf(oracle):
    rng = np.random.default_rng(7)
    v = _special_doubles(rng, 40000)
    n = (len(v) // 3) * 3
    g = v[:n].reshape(1, n // 3, 3)
    lp = v[3:9].copy()
    ep = v[11:17].copy()
    imu = v[20:26].copy()
    d = rng.integers(-2 ** 31, 2 ** 31 - 1, n // 3).astype(np.int32).reshape(1, -1)
    ours = nav.csv_format_frame(2 ** 40 + 7, g, lp, distances=d, imu=imu, ekf_pos=ep)
    want = oracle.csv_format_frame(2 ** 40 + 7, g, lp, distances=d, imu=imu, ekf_pos=ep)
    assert ours == want
    # and against an independent correctly rounded formatter (finite values only)
    first = ours.split(b"\n")[0].decode().split(",")
    assert first[3:6] == ["%.2f" % x for x in g[0, 0]]
    fin = np.isfinite(v[:n])
    got_cols = np.array([ln.split(b",")[3:6] for ln in ours.split(b"\n")[:-1]]).reshape(-1)
    for x, s in zip(v[:n][fin], got_cols[fin]):
        assert s.decode() == "%.2f" % x


def test_fixed2_nan_sign(oracle):
    g = np.array([[[float("nan"), -float("nan"), 1.0]]])
    assert nav.csv_format_frame(1, g, np.zeros(6)) == oracle.csv_format_frame(1, g, np.zeros(6))


def test_writer_defaults_and_header(oracle):
    rng = np.random.default_rng(3)
    g = rng.standard_normal((5, 33, 3)) * 3000.0
    lp = rng.standard_normal(6) * 100
    ours = nav.csv_format_frame(42, g, lp)
    assert ours == oracle.csv_format_frame(42, g, lp)
    assert ours.count(b"\n") == 5 * 33
    assert ours.split(b"\n")[0].split(b",")[6:13] == [b"0"] + [b"0.00"] * 6
    hdr = nav.load_library().nav_csv_header()
    assert hdr.count(b",") == 24 and hdr.endswith(b"EKF_yaw\n") and hdr.startswith(b"Timestamp,Row,Col,x,y,z,distance,")


def test_writer_buffer_too_small():
    import ctypes as C
    L = nav.load_library()
    g = np.zeros((8, 8, 3))
    buf = C.create_string_buffer(1000)
    lp = nav.binding.NavPos()
    assert L.nav_csv_format_frame(buf, len(buf), 1, 8, 8, g.ctypes.data, None, None, C.byref(lp), None) == 0


def _write(tmp_path, text, name="parsed_data.csv"):
    p = os.path.join(str(tmp_path), name)
    with open(p, "w", newline="") as f:
        f.write(text)
    return p


def _messy_csv(rng, rows, cols, n_frames, with_out_of_range=True):
    """Records in every number syntax fscanf accepts, some outside the image, frames of ragged coverage."""
    lines = ["frame,row,col,x,y,z,conf"]
    fmts = ["%d", "%.1f", "%.3f", "%.17g", "%e", "%+.2f", "%.25f", " %.4f", "%.0f."]
    for f in range(n_frames):
        frame_no = 10 + 3 * f
        for _ in range(rows * cols // 2 + 5):
            r, c = int(rng.integers(0, rows)), int(rng.integers(0, cols))
            if with_out_of_range and rng.random() < 0.05:
                r = int(rng.choice([-1, rows, rows + 7]))
            if with_out_of_range and rng.random() < 0.05:
                c = int(rng.choice([-3, cols + 1]))
            vals = rng.standard_normal(3) * 10.0 ** rng.integers(-3, 6)
            txt = []
            for v in vals:
                fm = fmts[int(rng.integers(0, len(fmts)))]
                txt.append(fm % (int(v) if fm == "%d" else v))
            lines.append(f"{frame_no},{r},{c},{txt[0]},{txt[1]},{txt[2]},{int(rng.integers(0, 255))}")
    return "\n".join(lines) + "\n"


@pytest.mark.parametrize("shape", [(8, 8), (5, 33)])
def test_reader_matches_reference_and_oracle(tmp_path, oracle, shape):
    rows, cols = shape
    rng = np.random.default_rng(rows * 100 + cols)
    path = _write(tmp_path, _messy_csv(rng, rows, cols, 6))
    frames, ts = nav.l9_csv_read(path, rows, cols, 10)
    rc, oframes, ots = oracle.l9_csv_read(path, rows, cols, 10)
    assert rc == 0 and len(frames) == 6
    assert np.array_equal(ts, ots) and list(ts) == [10, 13, 16, 19, 22, 25]
    assert frames.tobytes() == oframes.tobytes()
    ref = RefLib(rows, cols) if ref_available(f"{rows}x{cols}") else None
    rd = ref.l9_csv_read(path, 10) if ref is not None else None
    check_ref(f"l9_csv_read/{rows}x{cols}/timestamps", ts, rd and (lambda: rd[1]))
    check_ref(f"l9_csv_read/{rows}x{cols}/frames", frames, rd and (lambda: rd[0]))


def test_reader_integer_frames_config2(tmp_path, oracle):
    """BASELINE config 2's own input: 16x1800 integer millimetres written by synth.l9_csv."""
    seq = synth.l9_sequence(3)
    path = _write(tmp_path, synth.l9_csv(seq))
    frames, ts = nav.l9_csv_read(path, 16, 1800, 10)
    assert list(ts) == [0, 1, 2]
    assert np.array_equal(frames, np.trunc(seq))
    rd = RefLib(16, 1800).l9_csv_read(path, 10) if ref_available("16x1800") else None
    check_ref("l9_csv_read/16x1800/timestamps", ts, rd and (lambda: rd[1]))
    check_ref("l9_csv_read/16x1800/frames", frames, rd and (lambda: rd[0]))


def test_reader_edge_cases(tmp_path, oracle):
    # missing file: error with a message; the reference reports zero frames (main.c:80-83)
    with pytest.raises(nav.NavError):
        nav.l9_csv_read(os.path.join(str(tmp_path), "absent.csv"), 8, 8, 4)
    # header only / empty file: zero frames
    for text in ("", "frame,row,col,x,y,z,conf\n", "frame,row,col,x,y,z,conf"):
        f, ts = nav.l9_csv_read(_write(tmp_path, text), 8, 8, 4)
        assert len(f) == 0 and len(ts) == 0
    # parsing stops at the first malformed record, keeping what came before (fscanf != 7)
    text = "h\n1,0,0,1.5,2.5,3.5,9\n1,0,1,4,5,6,9\n1,0,2,oops,5,6,9\n2,0,0,7,8,9,9\n"
    p = _write(tmp_path, text)
    f, ts = nav.l9_csv_read(p, 8, 8, 4)
    rc, of, ots = oracle.l9_csv_read(p, 8, 8, 4)
    assert len(f) == 1 and f.tobytes() == of.tobytes() and f[0, 0, 1].tolist() == [4, 5, 6]
    # CRLF line ends, blank lines and a frame number that returns later start new frame slots
    text = "h\r\n5,0,0,1,2,3,9\r\n\r\n6,1,1,4,5,6,9\r\n5,2,2,7,8,9,9\r\n"
    p = _write(tmp_path, text)
    f, ts = nav.l9_csv_read(p, 8, 8, 4)
    rc, of, ots = oracle.l9_csv_read(p, 8, 8, 4)
    assert list(ts) == [5, 6, 5] == list(ots) and f.tobytes() == of.tobytes()
    # records whose row/col is outside the image do not start a frame (col == cols is rejected here; the
    # reference's `col > MAX_COLS` writes it one element out of bounds)
    text = "h\n1,0,8,1,2,3,9\n2,9,0,1,2,3,9\n3,0,0,1,2,3,9\n"
    f, ts = nav.l9_csv_read(_write(tmp_path, text), 8, 8, 4)
    assert list(ts) == [3]
    # more frames than the caller's buffer: an error instead of the reference's overrun of lidarData[10]
    text = "h\n" + "".join(f"{k},0,0,1,2,3,9\n" for k in range(6))
    with pytest.raises(nav.NavError):
        nav.l9_csv_read(_write(tmp_path, text), 8, 8, 4)
    # a header longer than the reference's 255-character fgets buffer: the tail is parsed as data
    text = "x" * 300 + "\n1,0,0,1,2,3,9\n"
    p = _write(tmp_path, text)
    f, _ = nav.l9_csv_read(p, 8, 8, 4)
    rc, of, _ = oracle.l9_csv_read(p, 8, 8, 4)
    assert len(f) == len(of) == 0


def test_read_then_write_round_trip(tmp_path, oracle):
    """CSV in -> frames -> CSV out -> same text a printf-based writer produces, and re-reading the x,y,z
    columns of that output gives the frames back to 2 decimals."""
    rng = np.random.default_rng(11)
    frames = np.round(rng.standard_normal((2, 5, 33, 3)) * 2000.0, 2)
    lines = ["frame,row,col,x,y,z,conf"]
    for f in range(2):
        for r in range(5):
            for c in range(33):
                lines.append("%d,%d,%d,%.2f,%.2f,%.2f,1" % (f, r, c, *frames[f, r, c]))
    path = _write(tmp_path, "\n".join(lines) + "\n")
    got, ts = nav.l9_csv_read(path, 5, 33, 4)
    assert got.tobytes() == frames.tobytes()
    out = nav.csv_format_frame(1, got[1], np.zeros(6))
    cols = np.array([ln.split(b",")[3:6] for ln in out.split(b"\n")[:-1]], dtype=np.float64)
    assert np.array_equal(cols.reshape(5, 33, 3), frames[1])


# ------------------------------------------------------------------ L5 / IMU JSON (src/main.c:12-75,130-178)
def _json_doc(rng, n, rows=8, cols=8):
    import json
    recs = []
    for f in range(n):
        recs.append({"time_main": 1000 + 7 * f, "extra": {"nested": [1, 2.5, "x", None, True]},
                     "distance": [int(v) for v in rng.integers(-5, 4000, rows * cols)],
                     "params": [float(v) for v in rng.normal(0, 1, 6)], "name": 'frame "%d"' % f})
    return json.dumps(recs, indent=1)


def test_json_readers_match_reference(tmp_path):
    rng = np.random.default_rng(5)
    synth_doc = synth.l5_json(6)                                    # config 1's own input file
    docs = {"synthetic": synth_doc, "random": _json_doc(rng, 9)}
    # shapes of trouble: a non-object element, a real inside distance, a short and an over-long distance
    # array, integer params (json_real_value gives 0.0), 5 params, a missing time, a repeated key
    docs["odd"] = ('[ {"time_main": 5, "distance": [1, 2.5, 3], "params": [1, 2.0, 3.5, 4.25, 5e-1, 6.0]},\n'
                   ' 17, {"distance": [%s], "params": [0.1, 0.2, 0.3, 0.4, 0.5]},\n'
                   ' {"time_main": 1.5, "distance": "none", "params": [0.5, 0.25, 0.125, 1.0, 2.0, -3.0],'
                   '  "time_main": 9, "distance": [7, 8]}, [] ]' % ", ".join(str(i) for i in range(80)))
    for name, doc in docs.items():
        p = _write(tmp_path, doc, name + ".json")
        d, ts = nav.l5_json_read(p, 8, 8, 100, fill=-77)
        prm, its = nav.imu_json_read(p, 100)
        if name == "synthetic":
            assert len(d) == 6 and np.array_equal(d[3], synth.l5_depth_frame(3))
        if name == "odd":
            assert len(d) == 5 and len(prm) == 3
            assert d[0].ravel()[:4].tolist() == [1, -77, 3, -77] and ts[0] == 5
            assert d[2].ravel()[:64].tolist() == list(range(64))
            assert d[3].ravel()[:3].tolist() == [7, 8, -77] and ts[3] == 9
            assert prm[0].tolist() == [0.0, 2.0, 3.5, 4.25, 0.5, 6.0] and prm[1].tolist() == [0.0] * 6
        ref = RefLib(8, 8) if ref_available("8x8") else None
        rd, rts = ref.l5_json_read(p, 100, fill=-77) if ref is not None else (None, None)
        rprm, rits = ref.imu_json_read(p, 100) if ref is not None else (None, None)
        check_ref(f"l5_json_read/{name}/distances", d, ref and (lambda: rd))
        check_ref(f"imu_json_read/{name}/params", prm, ref and (lambda: rprm))
        check_ref(f"imu_json_read/{name}/timestamps", its, ref and (lambda: rits))
        # a frame without an integer "time_main" keeps whatever the caller's buffer held: both start from 0 / -77
        check_ref(f"l5_json_read/{name}/timestamps", ts, ref and (lambda: rts), also=(np.where(ts == 0, -77, ts),))


def test_json_invalid_documents_read_nothing(tmp_path):
    for bad in ('[{"distance": [1, 2,]}]', '[{"distance": [1 2]}]', '[1, 2] x', '[{"a": 01}]', '[{"a": "\\q"}]', '',
                '[{"time_main": 1}', '[{"time_main": 99999999999999999999}]'):
        p = _write(tmp_path, bad, "bad.json")
        with pytest.raises(nav.NavError):
            nav.l5_json_read(p, 8, 8, 10)
        if ref_available("8x8"):
            rd, _ = RefLib(8, 8).l5_json_read(p, 10)
            assert len(rd) == 0
    # valid JSON that is not an array of frames: zero frames, no error
    for ok in ('{}', '[]', '3', ' "text" '):
        d, _ = nav.l5_json_read(_write(tmp_path, ok, "ok.json"), 8, 8, 10)
        assert len(d) == 0
    with pytest.raises(nav.NavError):
        nav.l5_json_read(_write(tmp_path, "[1,2,3]", "many.json"), 8, 8, 2)   # more frames than room
