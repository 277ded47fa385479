"""`python -m uwimageproc_b200.cli.chain` on JPEG files.  For every decoder x encoder x CLAHE choice, on a 4:2:0 and a 4:4:4
file: a one-file run writes the bytes a directory run writes for that file, and both are the bytes of the same pipeline
composed from Context calls (decode -> chain_dev / chain_auto_dev -> encode).  What each mode prints, for a fixed and an
automatic run, with a file whose entropy-coded data is cut short among the fixed run's inputs."""
import itertools

import pytest

from oracle import uwip_oracle as O
from test_jpeg_decoder_host import imencode

pytestmark = pytest.mark.gpu
SEED, W, H = 0x5EED0004, 160, 96
NOTE_BAD_DATA = "note: the file's entropy-coded data is bad; the frame was decoded as zeros"
NOTE_NAN = "note: the reference's exposure map is NaN for this frame (S = 0/0); the output is all zeros, as imwrite would store it"


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def _files():
    # synth frames 24 and 26: no NaN exposure map and a successful curve fit, fixed or automatic, from either decoder's pixels
    return {"a420.jpg": imencode(O.synth_frame(SEED, 24, W, H), 95, "420"),
            "b444.jpg": imencode(O.synth_frame(SEED, 26, W, H), 95, "444")}


def _cut_file():
    """test_gpu_jpeg_decoder.test_truncated_file_in_a_batch's file: the exact decoder sets flag 4 and decodes zeros."""
    b = imencode(O.synth_frame(SEED, 2, W, H), 95, "420")
    return b[:len(b) * 2 // 3]


def _dirs(tmp_path, files):
    src, dst, one = tmp_path / "src", tmp_path / "dst", tmp_path / "one"
    for d in (src, dst, one):
        d.mkdir()
    for name, data in files.items():
        (src / name).write_bytes(data)
    return src, dst, one


def _composed(ctx, data, decoder, encoder, auto, q=95):
    import torch

    w, h = ctx.jpeg_info(data)
    d_in = ctx.jpeg_decode_batch_dev([data]) if decoder == "exact" else ctx.jpeg_decode_dev(data)[None]
    d_out = torch.empty_like(d_in)
    if auto:
        ctx.chain_auto_dev(d_in, d_out, 1, w, h)
    else:
        ctx.chain_dev(d_in, d_out, 1, w, h)
    return ctx.jpeg_encode_batch_dev(d_out, q)[0] if encoder == "exact" else ctx.jpeg_encode_dev(d_out, w, h, q)


@pytest.mark.parametrize("decoder,encoder,auto", list(itertools.product(("nvjpeg", "exact"), ("nvjpeg", "exact"), (False, True))))
def test_one_file_equals_directory_and_composed_pipeline(ctx, tmp_path, decoder, encoder, auto):
    from uwimageproc_b200.cli import chain

    files = _files()
    src, dst, one = _dirs(tmp_path, files)
    opts = ["-decoder=" + decoder, "-encoder=" + encoder] + (["-aclahe=auto"] if auto else [])
    assert chain.main([str(src), str(dst)] + opts) == 0
    for name, data in files.items():
        assert chain.main([str(src / name), str(one / name)] + opts) == 0
        want = _composed(ctx, data, decoder, encoder, auto)
        assert (one / name).read_bytes() == want, name
        assert (dst / name).read_bytes() == want, name


def test_stdout_fixed(tmp_path, capsys):
    from uwimageproc_b200.cli import chain

    files = dict(_files(), **{"c_cut.jpg": _cut_file()})
    src, dst, one = _dirs(tmp_path, files)
    capsys.readouterr()
    assert chain.main([str(src), str(dst), "-decoder=exact"]) == 0
    assert capsys.readouterr().out.splitlines() == [
        "a420.jpg:", "saved %s" % (dst / "a420.jpg"),
        "b444.jpg:", "saved %s" % (dst / "b444.jpg"),
        "c_cut.jpg:", NOTE_BAD_DATA, NOTE_NAN, "saved %s" % (dst / "c_cut.jpg")]
    assert chain.main([str(src / "c_cut.jpg"), str(one / "c_cut.jpg"), "-decoder=exact"]) == 0
    assert capsys.readouterr().out.splitlines() == [NOTE_BAD_DATA, NOTE_NAN, "saved %s" % (one / "c_cut.jpg")]
    assert chain.main([str(src / "a420.jpg"), str(one / "a420.jpg"), "-decoder=exact"]) == 0
    assert capsys.readouterr().out.splitlines() == ["saved %s" % (one / "a420.jpg")]


def test_stdout_auto(tmp_path, capsys):
    """BS and CL are the oracle's ParametrosACLAHE on the V plane of histretch(cv2.imdecode(file))."""
    from uwimageproc_b200.cli import chain

    src, dst, one = _dirs(tmp_path, _files())
    capsys.readouterr()
    assert chain.main([str(src), str(dst), "-decoder=exact", "-aclahe=auto"]) == 0
    assert capsys.readouterr().out.splitlines() == [
        "a420.jpg: BS = 2 CL = 1", "saved %s" % (dst / "a420.jpg"),
        "b444.jpg: BS = 2 CL = 2", "saved %s" % (dst / "b444.jpg")]
    assert chain.main([str(src / "b444.jpg"), str(one / "b444.jpg"), "-decoder=exact", "-aclahe=auto"]) == 0
    assert capsys.readouterr().out.splitlines() == ["BS = 2 CL = 2", "saved %s" % (one / "b444.jpg")]
