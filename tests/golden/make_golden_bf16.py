"""Reference run in bfloat16 (tiny configuration, the inputs of tiny_prefill_decode.npz): pins the restatement's bf16 mode —
the "reference's own bf16 path" that the GPU parity tests use as their noise yardstick — against the unmodified reference.
PyTorch's CPU bf16 GEMMs take different kernels on different CPUs, and the results differ in the last bits (about 1 % of the
features by a few bf16 ulps), so the test's bit-exact feature check holds on hosts like the one this fixture was made on:
an x86 CPU with AMX-BF16 and AVX512-BF16.

    python tests/golden/make_golden_bf16.py        (build container only: needs /root/reference)
"""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import llava_oracle as O  # noqa: E402
from oracle import ref_shim  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    torch.set_grad_enabled(False)
    cfg = O.CONFIGS["tiny"]
    g = np.load(os.path.join(OUT, "tiny_prefill_decode.npz"))
    w = O.make_weights(cfg, seed=int(g["seed"]))
    model = ref_shim.build_reference_model(cfg, w, os.path.join(tempfile.mkdtemp(prefix="b2golden_bf16_"), "clip"),
                                           dtype=torch.bfloat16)
    ids, images = torch.from_numpy(g["input_ids"]), torch.from_numpy(g["images"]).to(torch.bfloat16)
    feats = model.encode_images(images)
    out = model(input_ids=ids, images=images, use_cache=True)
    # float32 holds every bfloat16 value exactly (float16 does not: its range and subnormals differ)
    np.savez_compressed(os.path.join(OUT, "tiny_bf16_prefill.npz"), image_features=feats.float().numpy(),
                        logits=out.logits.float().numpy(), seed=np.int64(int(g["seed"])))
    print("wrote tiny_bf16_prefill.npz")


if __name__ == "__main__":
    assert ref_shim.available(), "reference tree not found (this script only runs in the build container)"
    main()
