"""Record tests/golden/replays.json: what the UNMODIFIED reference produced in the live comparisons of
tests/test_oracle_golden.py and tests/test_gpu_sdl_shell.py, so that those tests compare with it in any checkout.

    python tests/golden/make_golden_replays.py [OUT]    # the shell part needs the built library and a CUDA device

    flythrough          sha256 of the 3 frames of the console-scripted flythrough (RGBA8 160x90)
    random_scenes       sha256 of the frames of the 18 random scenes
    shell_events        sha256 of the 16 frames the interactive shell hands to SDL under EVENTS, and its stdout
    shell_resize_cycle  sha256 and byte size of the compared frames under RESIZE_EVENTS with `cycle 3`

Where oracle/_ref is built the frames come from the reference itself.  Otherwise they come from the programs that
those tests found bit-identical to the reference on exactly these inputs: the oracle (oracle/hmap_oracle.c) for the
frames, the shell (host/hmap_sdl.cpp over libhmrm.so) for the shell runs.  `oracle_source` and `shell_source` in the
file say which.  Wherever oracle/_ref is built the tests keep comparing with the reference live as well.
"""
from __future__ import annotations

import json
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

import helpers as H  # noqa: E402
import oracle_lib as O  # noqa: E402
import scenes as S  # noqa: E402
import test_gpu_sdl_shell as SH  # noqa: E402
import test_oracle_golden as T  # noqa: E402


def reference_frame(scene, td: Path, binary=None, script=None):
    hm, cm = H.load_scene_maps(scene, O)
    O.write_png(td / "h.png", hm)
    O.write_png(td / "c.png", cm)
    kw = S.frame_kwargs(scene)
    cfg = O.config_text(kw, td / "h.png", td / "c.png", lum=scene["lum"])
    frames, _ = O.run_ref(cfg, scene["projection"], kw["width"], kw["height"], binary=binary, script=script)
    return frames


def oracle_part(td: Path) -> dict:
    if O.have_ref():
        script = ["pos %r %r %r hang %r" % (*s["pos"], s["hang_deg"]) for s in T.FLY_STATES]
        fly = reference_frame(T.FLY_SCENE, td, script=script)
        rand = [reference_frame(sc, td, binary=O.REF_BIN_O2)[0] for sc in T.random_scenes()]
        source = "the unmodified reference (oracle/_ref/hmap_ref, hmap_ref_O2)"
    else:
        fly = T.flythrough_oracle_frames(O, H.load_scene_maps(T.FLY_SCENE, O))
        rand = [H.oracle_render_scene(O, sc, H.load_scene_maps(sc, O))[0] for sc in T.random_scenes()]
        source = "the oracle, bit-identical to the unmodified reference on these scenes in the live comparison"
    return {"flythrough": [H.sha(f) for f in fly], "random_scenes": [H.sha(f) for f in rand], "oracle_source": source}


def shell_part(td: Path) -> dict:
    import __graft_entry__ as entry

    entry.build_product()
    if O.have_ref():
        binary, source = O.REF_BIN, "the unmodified reference (oracle/_ref/hmap_ref)"
    else:
        binary = SH.build_shell(td)
        source = "the shell (host/hmap_sdl.cpp), bit-identical to the unmodified reference under these scripts in the live comparison"
    out = {"shell_source": source}
    run = td / "events"
    run.mkdir()
    SH.write_inputs(O, run, "", SH.EVENTS)
    frames, stdout = SH.run_shell(binary, run, 16)
    out["shell_events"] = {"frame_sha256": [H.sha(f) for f in frames], "stdout": stdout}
    run = td / "resize_cycle"
    run.mkdir()
    SH.write_inputs(O, run, "cycle 3", SH.RESIZE_EVENTS)
    frames, _ = SH.run_shell(binary, run, 18)
    out["shell_resize_cycle"] = {"frame_sha256": {str(i): H.sha(frames[i]) for i in SH.RESIZE_COMPARED},
                                 "frame_size": {str(i): int(frames[i].size) for i in SH.RESIZE_COMPARED}}
    return out


if __name__ == "__main__":
    with tempfile.TemporaryDirectory(prefix="hmrm_gold_") as td:
        rec = {**oracle_part(Path(td)), **shell_part(Path(td))}
    out = Path(sys.argv[1]) if len(sys.argv) > 1 else HERE / "replays.json"
    out.write_text(json.dumps(rec, indent=1, sort_keys=True) + "\n")
    print(f"{out}: {rec['oracle_source']}; {rec['shell_source']}")
