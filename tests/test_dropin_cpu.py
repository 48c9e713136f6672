"""Drop-in check of the package-level boundary (INTEGRATION.md 1): the reference's own CLI module
video_super_resolution/scripts/inference_sr.py, unmodified, was run with `video_to_video` aliased to star_b200.video_to_video
and an in-memory clip (oracle/make_golden_reference.py); the calls it made into VideoToVideo_sr are stored in
tests/golden/reference_cli_calls.json and must bind to star_b200's signatures."""
import inspect
import json
import os
import types

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_cli_calls.json")


def test_reference_cli_runs_on_star_b200():
    from star_b200.video_to_video.video_to_video_model import VideoToVideo_sr
    calls = json.load(open(GOLD))
    init, test = calls["init"], calls["test"]
    opt = types.SimpleNamespace(**init["opt"])
    assert opt.model_path == "light_deg.pt" and not init["kwargs"]
    inspect.signature(VideoToVideo_sr.__init__).bind(None, opt, *init["args"])

    assert test["input_keys"] == ["target_res", "video_data", "y"] and test["kwargs"]["steps"] == 15
    video = test["input"]["video_data"]
    assert video["shape"][0] == 3 and test["input"]["target_res"] == [96, 128]
    inp = {"video_data": None, "y": test["input"]["y"], "target_res": tuple(test["input"]["target_res"])}
    bound = inspect.signature(VideoToVideo_sr.test).bind(None, inp, *test["args"], **test["kwargs"])
    assert bound.arguments["total_noise_levels"] == 900 and bound.arguments["solver_mode"] == "fast"
    # the reference's own post-processing turned the (1, 3, F, 96, 128) result into F frames of 96x128x3
    assert calls["saved"] == {"n": 3, "shape": [96, 128, 3]}
