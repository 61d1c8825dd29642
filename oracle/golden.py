"""The processor / Resampler goldens of tests/golden/processors/ (written by oracle/make_golden.py): one tensor dict stored as
numbered safetensors shards, each under 1 MB so that no single fixture file grows large."""
import glob
import os

PROCESSORS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "processors")
SHARD_BYTES = 900_000  # tensor payload per shard; the header adds a few KB


def save_processors(tensors, metadata, directory=PROCESSORS):
    """Write `tensors` (name -> tensor) as directory/part-NN.safetensors, packed in name order."""
    from safetensors.torch import save_file

    os.makedirs(directory, exist_ok=True)
    for old in glob.glob(os.path.join(directory, "part-*.safetensors")):
        os.remove(old)
    shards, cur, size = [], {}, 0
    for k in sorted(tensors):
        n = tensors[k].numel() * tensors[k].element_size()
        if cur and size + n > SHARD_BYTES:
            shards.append(cur)
            cur, size = {}, 0
        cur[k], size = tensors[k], size + n
    shards.append(cur)
    for i, shard in enumerate(shards):
        save_file(shard, os.path.join(directory, f"part-{i:02d}.safetensors"), metadata=metadata)
    return len(shards)


def load_processors(device="cpu", directory=PROCESSORS):
    """All shards merged back into one name -> tensor dict."""
    from safetensors import safe_open

    parts = sorted(glob.glob(os.path.join(directory, "part-*.safetensors")))
    assert parts, f"no golden shards under {directory}"
    out = {}
    for p in parts:
        with safe_open(p, "pt", device=str(device)) as f:
            for k in f.keys():
                assert k not in out, f"{k} stored twice"
                out[k] = f.get_tensor(k)
    return out
