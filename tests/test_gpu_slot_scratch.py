"""GPU: the encoder scratch of each frame-ring slot is one buffer that K3 (PNG), K4 (YUV) and K6 (JPEG) share.  Frames
in flight rotate the output kind so that every slot meets another kind on each pass and its scratch grows more than
once; every file and plane must be byte-equal to the same frame's output produced alone."""
import numpy as np
import pytest

import helpers as H
import scenes as S

pytestmark = pytest.mark.gpu

# per pixel, I420 planes < PNG scratch < JPEG 4:4:4 scratch: a slot that starts with YUV grows on each of its next two
# frames.  Frame i lands on ring slot (i + 1) % 4, so with three kinds each slot sees a different kind on every pass.
KINDS = ("yuv", "png", "jpeg")
FRAMES = 16
SCENE = dict(S.SCENE_BY_NAME["noise_lum"], width=640, height=360)


@pytest.fixture(scope="module")
def noise_renderer(hmrm):
    """A context of its own, so that its ring slots start without scratch, over the noise-like terrain of noise_lum:
    its frames barely compress, which fills most of the PNG scratch."""
    with hmrm.Renderer(0) as r:
        H.configure(r, SCENE, S.build_maps(SCENE["maps"], None))
        yield r


def test_slots_rotate_output_kinds_in_flight(hmrm, noise_renderer):
    r = noise_renderer
    W, Hh = SCENE["width"], SCENE["height"]
    frames = [H.product_frame(hmrm, r, dict(SCENE, pos=(-0.4 + 0.03 * i, 0.5 - 0.02 * i, 2.2), hang_deg=-45.0 - 5.0 * i))
              for i in range(FRAMES)]
    kinds = [KINDS[i % len(KINDS)] for i in range(FRAMES)]
    bufs = []
    for k in kinds:
        n = {"yuv": hmrm.yuv420_bytes(W, Hh), "png": hmrm.png_bound(W, Hh, 4),
             "jpeg": hmrm.jpeg_bound(W, Hh, hmrm.JPEG_444)}[k]
        bufs.append((hmrm.pinned_empty((n,)), hmrm.pinned_empty((1,), dtype=np.uint64)))

    # every frame is enqueued before the first wait
    for k, f, (out, size) in zip(kinds, frames, bufs):
        if k == "yuv":
            r.render_yuv420_async(f, out, hmrm.YUV_BT709)
        elif k == "png":
            r.render_png_async(f, out, size)
        else:
            r.render_jpeg_async(f, out, size, 100, hmrm.JPEG_444)
    r.wait()
    got = [out.tobytes() if k == "yuv" else out[:int(size[0])].tobytes() for k, (out, size) in zip(kinds, bufs)]

    for i, (k, f) in enumerate(zip(kinds, frames)):
        if k == "yuv":
            want = b"".join(p.tobytes() for p in r.render_yuv420(f, hmrm.YUV_BT709))
        elif k == "png":
            want = r.render_png(f)
        else:
            want = r.render_jpeg(f, 100, hmrm.JPEG_444)
        assert got[i] == want, f"frame {i} ({k})"
