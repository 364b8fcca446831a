"""What the native executors pack, pinned against a stored fixture.

For the tiny FLUX / WAN / Z-Image / UNet models (seed 0, bf16, CPU) the fixture holds the packed weight table (key
order, shapes, dtypes, SHA-256 of the bytes), one activation workspace per DiT family (keys, shapes, dtypes), a SHA-256
of the fp32 RoPE table and the signatures of the public step entry points.  Packed checkpoints and NVLink replication
match weights by these keys, the sequence-parallel drivers use the workspace keys, and callers hold on to these
signatures, so a change to any of them has to be deliberate.

``python tests/test_executor_packing.py --write`` regenerates ``tests/golden/executor_packing.json``.
"""
import hashlib
import inspect
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden", "executor_packing.json")
FAMILIES = ("flux", "wan", "zimage", "unet")
ENTRY_POINTS = ("forward", "forward_shard", "shard_graph_handle", "denoise_step", "_prep")


def _sha(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().cpu().contiguous().reshape(-1).view(torch.uint8).numpy().tobytes()).hexdigest()


def _describe(v, with_hash: bool):
    if isinstance(v, torch.Tensor):
        d = [list(v.shape), str(v.dtype)]
        return d + [_sha(v)] if with_hash else d
    if isinstance(v, (list, tuple)):
        return [_describe(x, with_hash) for x in v]
    if isinstance(v, dict):
        return {str(k): _describe(x, with_hash) for k, x in v.items()}
    return repr(v)


def _build(family: str):
    from comfyui_parallelanything_b200.models import flux, unet, wan, zimage
    torch.manual_seed(0)
    if family == "flux":
        from comfyui_parallelanything_b200.exec.flux_exec import FluxExecutor
        return FluxExecutor(flux.Flux(flux.flux_tiny_params()).to(torch.bfloat16), "cpu"), (1, 16, 16, 8)
    if family == "wan":
        from comfyui_parallelanything_b200.exec.wan_exec import WanExecutor
        return WanExecutor(wan.WanModel(wan.wan_tiny_params()).to(torch.bfloat16), "cpu"), (1, 2, 8, 8, 8)
    if family == "zimage":
        from comfyui_parallelanything_b200.exec.zimage_exec import ZImageExecutor
        return ZImageExecutor(zimage.ZImageModel(zimage.zimage_tiny_params()).to(torch.bfloat16), "cpu"), (1, 8, 8, 8)
    from comfyui_parallelanything_b200.exec.unet_exec import UNetExecutor
    return UNetExecutor(unet.UNetModel(**unet.mini_sdxl_config()).to(torch.bfloat16), "cpu"), None


def record(family: str) -> dict:
    from comfyui_parallelanything_b200.exec.pack_cache import packed_table
    ex, geometry = _build(family)
    table = packed_table(ex)
    rec = {"packed_keys": list(table), "packed": {k: _describe(v, True) for k, v in table.items()},
           "signatures": {m: str(inspect.signature(getattr(ex, m))) for m in ENTRY_POINTS if hasattr(ex, m)}}
    if geometry is not None:
        ws = ex.workspace(*geometry)
        rec["workspace_keys"] = list(ws)
        rec["workspace"] = {k: _describe(v, False) for k, v in ws.items()}
        rec["rope_sha256"] = _sha(ws["ROPE"])
    return rec


@pytest.mark.parametrize("family", FAMILIES)
def test_executor_packing_matches_fixture(family):
    with open(GOLDEN) as f:
        want = json.load(f)[family]
    got = json.loads(json.dumps(record(family)))          # tuples -> lists, as stored
    assert got["packed_keys"] == want["packed_keys"]
    for k in want["packed"]:
        assert got["packed"][k] == want["packed"][k], k
    assert got["signatures"] == want["signatures"]
    assert got.get("workspace_keys") == want.get("workspace_keys")
    assert got.get("workspace") == want.get("workspace")
    assert got.get("rope_sha256") == want.get("rope_sha256")
    assert got == want


if __name__ == "__main__":
    if sys.argv[1:] != ["--write"]:
        sys.exit("usage: python tests/test_executor_packing.py --write")
    data = {fam: record(fam) for fam in FAMILIES}
    with open(GOLDEN, "w") as f:
        json.dump(data, f, indent=1, sort_keys=False)
        f.write("\n")
    print(f"wrote {GOLDEN}")
