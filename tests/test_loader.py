""".rts / .ppm / .bmp host code vs the reference's read() (oracle/_ref) and the C restatement."""
import os
import struct

import numpy as np
import pytest

import dogeray_b200 as drb
from dogeray_b200 import synth
from oracle import restated
from conftest import HAVE_REF, SAMPLES, all_sample_scenes, needs_ref, sample

# files whose junk / legacy lines leave fields indeterminate in the reference (SURVEY App. A, B.9)
UB_FILES = {"HIGH.rts", "light.rts", "rough.rts"}


def settings_vector(st):
    return np.array([st.cam[0], st.cam[1], st.cam[2], st.aperture, st.look[0], st.look[1], st.look[2], st.focus, st.fov,
                     st.max_depth, st.spp, st.bg_intensity, st.backtex, st.width, st.height], np.float32)


def compare_objects(ours, theirs, ncols):
    """bit-exact on every column the line actually had"""
    def eq(a, b):
        return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))
    col_of = [("pos", "pos", 0), ("col", "col", 4), ("dim", "dim", 9), ("rot", "rot", 13), ("norm", "norm", 16), ("n1", "n1", 19),
              ("n2", "n2", 22), ("n3", "n3", 25)]
    for mine, ref_name, first in col_of:
        m = ncols >= first + 3
        assert eq(ours[mine][m], theirs[ref_name][m]), mine
    m = ncols >= 4; assert np.array_equal(ours["type"][m], theirs["type"][m])
    m = ncols >= 8; assert eq(ours["add_y"][m], theirs["addional"][m][:, 1])
    m = ncols >= 9; assert eq(ours["add_x"][m], theirs["addional"][m][:, 0])
    m = ncols >= 13; assert np.array_equal(ours["mat"][m], theirs["mat"][m])
    for k, first in (("t1", 28), ("t2", 30), ("t3", 32)):
        m = ncols >= first + 2
        assert eq(ours[k][m], theirs[k][m][:, :2]), k
    m = ncols >= 35; assert np.array_equal(ours["smooth"][m] != 0, theirs["smooth"][m] != 0)
    m = ncols >= 36; assert np.array_equal(ours["checker"][m] != 0, theirs["tex"][m] != 0)
    assert np.array_equal(ours["texnum"], theirs["texnum"])
    assert np.array_equal(ours["rtexnum"], theirs["rtexnum"])


@needs_ref
@pytest.mark.parametrize("name", all_sample_scenes())
def test_loader_matches_reference_read(ref, name):
    hs = drb.HostScene.load(sample(name), SAMPLES)
    if os.path.getsize(sample(name)) == 0:
        assert hs.num_objects == 0
        return
    n = ref.load(sample(name), SAMPLES)
    assert n == hs.num_objects + 1                      # getnum returns lines + 1 (kernel.cu:1158)
    assert np.array_equal(settings_vector(hs.settings), ref.get_settings()[:15])
    assert [os.path.basename(p) for p in hs.texture_paths] == [os.path.basename(p) for p in ref.texture_paths()]
    ours = hs.objects()
    if name in UB_FILES:
        good = ours["ncols"] >= 13
        compare_objects(ours[good], ref.objects()[good], ours["ncols"][good])
    else:
        compare_objects(ours, ref.objects(), ours["ncols"])


@needs_ref
def test_texture_name_lookup_quirks():
    # names with capitals never resolve: the candidate is lower-cased, the query is not (kernel.cu:1176-1178)
    hs = drb.HostScene.load(sample("test6.rts"), SAMPLES)
    assert hs.settings.backtex == -1 or hs.num_objects >= 0
    hs = drb.HostScene.load(sample("bolter2.blend.rts"), SAMPLES)
    tp = [os.path.basename(p) for p in hs.texture_paths]
    assert tp[hs.settings.backtex] == "env.ppm"
    o = hs.objects()
    assert set(np.unique(o["texnum"])) <= {-1, tp.index("boltersmall.ppm")}
    assert (o["texnum"] >= 0).any()
    text = b"*,0,0,2,0.01,0,0,0,3,45,5,1,1,UV_Checker.ppm\n"
    assert drb.HostScene.parse(text, SAMPLES).settings.backtex == -1


def test_edge_cases_empty_and_settings_only():
    hs = drb.HostScene.parse(b"")
    assert hs.num_objects == 0 and hs.settings.as_dict() == drb.default_settings().as_dict()
    hs = drb.HostScene.parse(b"/comment\n*,1,2,3,0.5,4,5,6,7,60.9,12.000000,3,0.25,no,640,480\n")
    s = hs.settings
    assert hs.num_objects == 0 and list(s.cam) == [1, 2, 3] and s.aperture == 0.5 and list(s.look) == [4, 5, 6]
    assert s.focus == 7 and s.fov == 60 and s.max_depth == 12 and s.spp == 3 and s.bg_intensity == 0.25       # stoi("60.9") == 60
    assert s.backtex == -1 and (s.width, s.height) == (640, 480)


def test_edge_cases_short_lines_crlf_blank_and_random_token():
    text = (b"1,2,3,0,0.5,0.6,0.7,0.1,0,4,0,0,3\r\n"           # 13-column sphere, CRLF
            b"\n"                                                # blank line: skipped (the reference throws)
            b"0,0,0,2,1,1,1,0,0,1,0,0,0,0,1,0\n"                 # 16-column triangle
            b"00\n"                                              # junk line as in samples/HIGH.rts
            b"r,0,0,2,1,1,1,0,0,1,0,0,0,0,1,0")                  # 'r' token, no trailing newline
    hs = drb.HostScene.parse(text)
    o = hs.objects()
    assert hs.num_objects == 4 and list(o["ncols"]) == [13, 16, 1, 16]
    assert o["type"][0] == 0 and o["mat"][0] == 3 and o["dim"][0][0] == 4
    assert hs.num_skipped == 2                                   # the blank line and the junk object
    assert 0.0 <= o["pos"][3][0] < 1.0
    assert o["pos"][3][0] == drb.HostScene.parse(text).objects()["pos"][3][0]     # deterministic
    assert list(o["norm"][1]) == [-2, -3, -20] and list(o["t1"][1]) == [0, 1] and o["texnum"][1] == -1


def test_parse_errors_are_reported_not_thrown():
    for bad in (b"1,2,,2\n", b"1,2,3,x\n", b"*,1,2,zz\n"):
        with pytest.raises(drb.DogerayError) as e:
            drb.HostScene.parse(bad)
        assert e.value.status == drb.ERR_PARSE


def test_large_parse_is_parallel_and_ordered(tmp_path):
    objs, st = synth.heightfield_scene(n=120)          # 28 800 triangles -> several parser threads
    p = str(tmp_path / "big.rts")
    drb.write_rts(p, st, objs)
    back = drb.HostScene.load(p).objects()
    assert len(back) == len(objs)
    for k in ("pos", "dim", "rot", "col", "norm", "n1", "n2", "n3", "t1", "t2", "t3"):
        assert np.allclose(back[k], objs[k], atol=1e-6), k       # %f keeps 6 decimals
    assert np.array_equal(back["mat"], objs["mat"]) and np.array_equal(back["type"], objs["type"])
    r = restated.Restated(p)
    assert r.num_objects == len(objs)


def _numbered_scene(nlines, seed):
    """text whose object line k carries k in its first column, with comments, blank lines, CRLF endings, ragged line
    lengths and one settings line sprinkled in; returns (text, expected first-column values, blank count, first blank line)"""
    rng = np.random.default_rng(seed)
    out, expect, blanks, first_blank = [], [], 0, None
    kinds = rng.integers(0, 100, nlines)
    for i in range(nlines):
        k = kinds[i]
        if k < 3:
            out.append(b"/ comment %d" % i + b" x" * int(rng.integers(0, 40)))
        elif k < 5:
            out.append(b"")
            blanks += 1
            first_blank = i + 1 if first_blank is None else first_blank
        elif i == nlines // 2:
            out.append(b"*,1,2,3,0.01,0,0,0,3,45,7,9,1,no,64,32")
        else:
            v = len(expect)
            cols = [b"%d" % v, b"1", b"2", b"2", b"0.5", b"0.5", b"0.5", b"0", b"0", b"1", b"0", b"0", b"0", b"0", b"1", b"0"]
            cols += [b"0.25"] * int(rng.integers(0, 20))                # ragged: 16..35 columns
            out.append(b",".join(cols) + (b"\r" if k % 2 else b""))
            expect.append(v)
    return b"\n".join(out), np.array(expect, np.float32), blanks, first_blank


def test_parallel_parse_numbers_lines_like_a_sequential_pass(tmp_path):
    """> 8 MiB of text: every byte range, chunk boundary and prefix sum of the parallel parser is exercised; object
    order, skipped count, the first warning and the line number of an injected error must be the sequential ones"""
    text, expect, blanks, first_blank = _numbered_scene(150_000, seed=2)
    assert len(text) > 8 << 20
    for tail in (b"", b"\n"):                                            # with and without a final newline
        hs = drb.HostScene.parse(text + tail)
        o = hs.objects()
        assert len(o) == len(expect) and np.array_equal(o["pos"][:, 0], expect)
        assert hs.num_skipped == blanks and ("line %d: blank line skipped" % first_blank).encode() in drb._lib.drb_last_error()
        assert hs.settings.max_depth == 7 and hs.settings.spp == 9 and (hs.settings.width, hs.settings.height) == (64, 32)
    p = str(tmp_path / "n.rts")
    open(p, "wb").write(text)
    assert np.array_equal(drb.HostScene.load(p).objects().view(np.uint8), o.view(np.uint8))
    # an error far into the file is reported with its own line number; of two errors the earlier one wins
    lines = text.split(b"\n")
    bad = [i for i, l in enumerate(lines) if l[:1] not in (b"", b"/", b"*")]
    first, second = bad[len(bad) // 3], bad[2 * len(bad) // 3]
    for i in (second, first):
        lines[i] = lines[i].replace(b",2,0.5,", b",2,oops,", 1)
        with pytest.raises(drb.DogerayError) as e:
            drb.HostScene.parse(b"\n".join(lines))
        assert e.value.status == drb.ERR_PARSE and "line %d column 4" % (i + 1) in str(e.value)
    # an unrenderable object is a warning only when no blank line came first
    clean = b"\n".join(l for l in text.split(b"\n") if l != b"")
    cl = clean.split(b"\n")
    idx = [i for i, l in enumerate(cl) if l[:1] not in (b"/", b"*")][1000]
    cl[idx] = cl[idx].replace(b",1,2,2,", b",1,2,7,", 1)                  # type 7: kept, not renderable
    hs = drb.HostScene.parse(b"\n".join(cl))
    assert hs.num_skipped == 1 and ("line %d: object with type 7" % (idx + 1)).encode() in drb._lib.drb_last_error()
    assert hs.num_objects == len(expect)


def test_rts_writer_is_exporter_format(tmp_path):
    objs, st = synth.heightfield_scene(n=2)
    p = str(tmp_path / "w.rts")
    drb.write_rts(p, st, objs)
    lines = open(p).read().splitlines()
    assert lines[0].startswith("/") and lines[1].startswith("*,") and len(lines[1].split(",")) == 16
    assert all(len(l.split(",")) == 38 for l in lines[2:]) and len(lines) == 2 + len(objs)
    hs = drb.HostScene.load(p)
    assert np.array_equal(settings_vector(hs.settings), settings_vector(st))


def test_ppm_reader(tmp_path):
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    p = str(tmp_path / "t.ppm")
    with open(p, "wb") as f:
        f.write(b"P6\n# a comment\n7 5\n255\n" + img.tobytes())
    rgba = drb.read_ppm(p)
    assert rgba.shape == (5, 7, 4) and np.array_equal(rgba[..., :3], img) and (rgba[..., 3] == 0).all()
    with open(p, "wb") as f:
        f.write(b"P6\n7 5\n255\n" + img.tobytes()[:-3])
    with pytest.raises(drb.DogerayError):
        drb.read_ppm(p)


@needs_ref
def test_ppm_reader_on_shipped_textures():
    for name in ("a.ppm", "env.ppm", "test.PPM"):
        rgba = drb.read_ppm(sample(name))
        raw = open(sample(name), "rb").read()
        hdr = raw.split(b"\n", 3)
        w, h = (int(v) for v in hdr[1].split())
        assert rgba.shape == (h, w, 4)
        assert np.array_equal(rgba[..., :3].reshape(-1), np.frombuffer(hdr[3], np.uint8)[: w * h * 3])


def test_bmp_layout_is_sdl_savebmp_v4(tmp_path):
    rng = np.random.default_rng(2)
    img = rng.integers(0, 256, (3, 4, 3), dtype=np.uint8)
    p = str(tmp_path / "o.bmp")
    drb.write_bmp(p, img)
    b = open(p, "rb").read()
    assert b[:2] == b"BM" and len(b) == 122 + 4 * 3 * 4
    size, _, off = struct.unpack_from("<IiI", b, 2)
    assert size == len(b) and off == 122
    hsz, w, h, planes, bpp, comp, isz = struct.unpack_from("<IiiHHII", b, 14)
    assert (hsz, w, h, planes, bpp, comp, isz) == (108, 4, 3, 1, 32, 3, 48)         # SURVEY.md App. C.1
    assert struct.unpack_from("<IIII", b, 14 + 40) == (0x00FF0000, 0x0000FF00, 0x000000FF, 0xFF000000)
    assert struct.unpack_from("<I", b, 14 + 56)[0] == 0x57696E20
    px = np.frombuffer(b[122:], np.uint8).reshape(3, 4, 4)[::-1]                     # bottom-up rows, B G R A
    assert np.array_equal(px[..., 2], img[..., 0]) and np.array_equal(px[..., 1], img[..., 1]) and np.array_equal(px[..., 0], img[..., 2])
    assert (px[..., 3] == 255).all()


def test_bmp_header_equals_the_reference_screenshots_byte_for_byte(tmp_path):
    """tests/golden/bmp_headers.json holds the first 122 bytes of every images/*.bmp the reference ships (SDL_SaveBMP,
    kernel.cu:2505-2513): a file of the same size must start with exactly those bytes, and alpha is 255 throughout"""
    import json
    here = os.path.dirname(os.path.abspath(__file__))
    with open(os.path.join(here, "golden", "bmp_headers.json")) as f:
        golden = json.load(f)
    assert "bolter2.blend.rts.bmp" in golden and len(golden) >= 13
    done = set()
    for name, g in golden.items():
        assert g["pixel_offset"] == 122 and g["alpha_values"] == [255]
        key = (g["width"], g["height"])
        if key in done:
            continue
        done.add(key)
        img = np.zeros((g["height"], g["width"], 3), np.uint8)
        img[0, 0] = (1, 2, 3)
        p = str(tmp_path / "o.bmp")
        drb.write_bmp(p, img)
        b = open(p, "rb").read()
        assert len(b) == g["file_size"], name
        assert b[:122].hex() == g["header_hex"], name
    assert (1280, 720) in done and len(done) >= 3


SCREENSHOT = os.path.join(os.path.dirname(SAMPLES), "bolter2.blend.rts.bmp")


@pytest.mark.skipif(not os.path.exists(SCREENSHOT), reason="the reference's screenshot is staged into oracle/_ref by oracle/make_ref.py")
def test_bmp_writer_reproduces_a_reference_screenshot_file(tmp_path):
    """decode images/bolter2.blend.rts.bmp to top-down RGB and write it back: the file must come out byte-identical"""
    ref = open(SCREENSHOT, "rb").read()
    w, h = struct.unpack_from("<ii", ref, 18)
    px = np.frombuffer(ref[122:], np.uint8).reshape(h, w, 4)[::-1]            # bottom-up rows, B G R A
    rgb = np.ascontiguousarray(px[..., [2, 1, 0]])
    p = str(tmp_path / "again.bmp")
    drb.write_bmp(p, rgb)
    assert open(p, "rb").read() == ref


def test_ppm_writer_and_tonemap(tmp_path):
    acc = np.array([[[0.0, 0.5, 1.0], [2.0, -1.0, float("nan")]]], np.float32) * 4        # sum over 4 samples
    out = drb.tonemap(acc, 4)
    assert out.tolist() == [[[0, 127, 255], [255, 0, 0]]]                                 # trunc, clamp, NaN -> 0 (kernel.cu:1083-1085, 2287)
    p = str(tmp_path / "o.ppm")
    drb.write_ppm(p, out)
    assert open(p, "rb").read() == b"P6\n2 1\n255\n" + out.tobytes()
