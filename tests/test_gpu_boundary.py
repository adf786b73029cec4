"""-m gpu: the reference's caller sequence (inference.py:37-59) against this repo's ``vlm_fo1`` mirror and a fabricated
random-init checkpoint directory: load_pretrained_model -> prepare_inputs -> model.generate -> tokenizer.decode ->
extract_predictions_to_bboxes -> draw_bboxes_and_save, with the script's own defaults (device="cuda", max_tokens=4096,
torch.inference_mode).  The checkpoint is reduced-depth (real widths) so fabrication stays small; a full-depth directory
is produced the same way by ``vlm-fo1_b200/fabricate.py``."""
import os

import numpy as np
import pytest
import torch
from PIL import Image

pytestmark = pytest.mark.gpu


def _fabricate(root, num_hidden_layers):
    from importlib import import_module
    import fo1_b200  # noqa: F401
    E = import_module("vlm-fo1_b200.engine"); FB = import_module("vlm-fo1_b200.fabricate")
    cfg = E.EngineConfig()
    cfg.vit = dict(cfg.vit, depth=2, fullatt_block_indexes=[0, 1])
    cfg.davit = dict(cfg.davit, depths=[1, 1, 1, 1])
    cfg.llm = dict(cfg.llm, num_hidden_layers=num_hidden_layers)
    return FB.fabricate_checkpoint(os.path.join(str(root), "resources", "VLM-FO1_Qwen2.5-VL-3B-v01"), cfg, seed=0, device="cuda")


def _inference_py(img_path, model_path, out_path, max_new_tokens=None):
    """The statements of inference.py, unchanged apart from the three paths; ``max_new_tokens`` optionally bounds the
    script's max_tokens=4096.  Returns (model, generation_kwargs, output_ids, outputs, bboxes)."""
    from detect_tools.upn import UPNWrapper  # noqa: F401
    from vlm_fo1.model.builder import load_pretrained_model
    from vlm_fo1.mm_utils import prepare_inputs, draw_bboxes_and_save, extract_predictions_to_bboxes
    from vlm_fo1.task_templates import OD_template
    bbox_list = [[161.0, 11.0, 292.0, 127.0], [268.0, 61.0, 428.0, 226.0], [12.0, 100.0, 140.0, 227.0], [205.0, 188.0, 332.0, 320.0],
                 [326.0, 202.0, 478.0, 357.0], [136.0, 106.0, 269.0, 233.0], [25.0, 206.0, 200.0, 383.0]]
    messages = [{"role": "user", "content": [{"type": "image_url", "image_url": {"url": img_path}},
                                             {"type": "text", "text": OD_template.format("orange")}], "bbox_list": bbox_list}]
    tokenizer, model, image_processors = load_pretrained_model(model_path)
    generation_kwargs = prepare_inputs(model_path, model, image_processors, tokenizer, messages,
                                       max_tokens=4096, top_p=0.05, temperature=0.0, do_sample=False)
    if max_new_tokens is not None:
        generation_kwargs["max_new_tokens"] = max_new_tokens
    with torch.inference_mode():
        output_ids = model.generate(**generation_kwargs)
        outputs = tokenizer.decode(output_ids[0, generation_kwargs["inputs"].shape[1]:]).strip()
    bboxes = extract_predictions_to_bboxes(outputs, bbox_list)
    draw_bboxes_and_save(image=Image.open(img_path).convert("RGB"), fo1_bboxes=bboxes, output_path=out_path)
    return model, generation_kwargs, output_ids, outputs, bboxes


def test_inference_py_call_sequence(tmp_path):
    model_path = _fabricate(tmp_path, 2)
    img_path = str(tmp_path / "demo_image.jpg")
    Image.fromarray(np.random.default_rng(0).integers(0, 256, (399, 500, 3), dtype=np.uint8)).save(img_path)
    out_path = str(tmp_path / "vlm_fo1_result.jpg")
    # (the test bounds the length; a random-init model never emits <|im_end|>)
    model, generation_kwargs, output_ids, outputs, bboxes = _inference_py(img_path, model_path, out_path, max_new_tokens=24)
    # ---- contract checks ----
    P = generation_kwargs["inputs"].shape[1]
    assert output_ids.dim() == 2 and output_ids.shape[0] == 1 and P < output_ids.shape[1] <= P + 24
    assert torch.equal(output_ids[0, :P].cpu(), generation_kwargs["inputs"][0].cpu())      # callers slice at inputs.shape[1]
    assert isinstance(outputs, str) and isinstance(bboxes, dict) and os.path.exists(out_path)
    # determinism + stop handling through the same surface: stop on the 3rd generated id
    new = output_ids[0, P:].tolist()
    model.default_stop_ids = [new[2]]
    again = model.generate(**generation_kwargs)
    assert again[0, P:].tolist() == new[: new.index(new[2]) + 1]


def test_inference_py_call_sequence_at_script_defaults(tmp_path, monkeypatch):
    """The same statements run as inference.py runs them: from a working directory laid out like the reference's
    (./resources/<checkpoint>, ./demo/demo_image.jpg), with the script's relative paths and its unbounded max_tokens=4096
    (a random-init model never emits <|im_end|>)."""
    _fabricate(tmp_path, 1)
    os.makedirs(tmp_path / "demo")
    Image.fromarray(np.random.default_rng(0).integers(0, 256, (399, 500, 3), dtype=np.uint8)).save(str(tmp_path / "demo" / "demo_image.jpg"))
    monkeypatch.chdir(tmp_path)
    _, generation_kwargs, output_ids, outputs, bboxes = _inference_py("demo/demo_image.jpg", "./resources/VLM-FO1_Qwen2.5-VL-3B-v01",
                                                                      "demo/vlm_fo1_result.jpg")
    P = generation_kwargs["inputs"].shape[1]
    assert output_ids.shape[0] == 1 and P < output_ids.shape[1] <= P + 4096
    assert isinstance(outputs, str) and isinstance(bboxes, dict)
    assert os.path.exists(tmp_path / "demo" / "vlm_fo1_result.jpg")
