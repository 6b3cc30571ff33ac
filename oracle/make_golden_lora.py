#!/usr/bin/env python
"""Turns the reference's shipped, trained LoRA adapters (lora_weights1/lora_weights.pkl, the only real weight artefact of
the repository; SURVEY.md F5) into a numeric fixture: tests/golden/lora_weights1_arrays.npz, one array per
(layer, projection, A | B) + the metadata fields.  The arrays are stored as float16 in a compressed archive, which keeps
the fixture under 1 MB (fp32 would be 1.5 MB); the rounding moves no value by more than 3.1e-5, far below the trained
magnitudes the tests rely on.  TEST INFRASTRUCTURE ONLY; needs a checkout of the reference repository.

    python oracle/make_golden_lora.py --reference <checkout of the reference>

tests rebuild a pickle in the reference's layout (save_lora, test.py:642-684) from these arrays and load it through the
product's `load_lora` (test.py:695-735), so that the towers are held to the oracle with REAL trained adapter magnitudes
(|A| <= 0.05, |B| <= 0.012) and the encoder='both' layer mapping (text blocks = layer_0..11, vision blocks = layer_12..23).
"""
import argparse
import json
import os
import pickle

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of the reference repository")
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "lora_weights1_arrays.npz"))
    a = ap.parse_args()
    with open(os.path.join(a.reference, "lora_weights1", "lora_weights.pkl"), "rb") as f:
        d = pickle.load(f)
    arrays = {"metadata_json": np.frombuffer(json.dumps(d["metadata"]).encode(), dtype=np.uint8)}
    for layer, projs in d["weights"].items():
        for proj, ab in projs.items():
            for name, arr in ab.items():
                arrays[f"{layer}/{proj}/{name}"] = np.asarray(arr, dtype=np.float32).astype(np.float16)
    np.savez_compressed(a.out, **arrays)
    print(f"wrote {a.out}: {len(arrays) - 1} arrays, metadata {d['metadata']}")


if __name__ == "__main__":
    main()
