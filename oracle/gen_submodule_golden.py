"""Golden vectors for tests/test_submodules_gpu.py: the UNMODIFIED reference sub-module classes (FactorEncoder, AlphaLayer,
BetaLayer, FactorDecoder, AttentionLayer, FactorPredictor of the original project's module.py), loaded with the state_dict of
our seeded modules and called on the test's inputs, on the CPU.

Test infrastructure only; needs a checkout of the original project:

    python oracle/gen_submodule_golden.py <original project directory>

Writes tests/golden/submodules_reference.npz: per test shape, every output the test compares, float32 as the reference
computes it; outputs with more than REF_ROWS rows are kept for the fixed row sample test_submodules_gpu.ref_rows()."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.join(HERE, "..", "tests")


def main():
    if len(sys.argv) != 2 or not os.path.isfile(os.path.join(sys.argv[1], "module.py")):
        raise SystemExit(__doc__)
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))
    sys.path.insert(0, TESTS)
    import module as ref                      # noqa: E402  (the reference's module.py, unmodified)
    import test_submodules_gpu as T           # noqa: E402  (shapes, seeds and inputs of the test)

    torch.set_num_threads(1)
    blob = {}
    for shape in T.SHAPES:
        N, H, K, M = (shape[k] for k in "NHKM")
        _, enc, dec, pred = T._modules(H, K, M)
        e, y = T._inputs(N, H)
        zmu, zsg, eps = T._decoder_noise(N, K)
        out = {}
        with torch.no_grad():
            r = ref.FactorEncoder(K, M, H)
            r.load_state_dict(enc.state_dict())
            out["enc_mu"], out["enc_sigma"] = r(e, y)
            r = ref.FactorDecoder(ref.AlphaLayer(H), ref.BetaLayer(H, K))
            r.load_state_dict(dec.state_dict())
            out["alpha_mu"], out["alpha_sigma"] = r.alpha_layer(e)
            out["beta"] = r.beta_layer(e)
            r.reparameterize = lambda mu, sigma: mu + eps.view(-1, 1) * sigma         # the test injects the same eps
            out["decoder_y"] = r(e, zmu.clone(), zsg.clone())
            r = ref.FactorPredictor(H, K)
            r.load_state_dict(pred.state_dict())
            r.eval()
            out["predictor_mu"], out["predictor_sigma"] = r(e)
            out["context0"] = r.attention_layers[0](e)
        rows = T.ref_rows(N)
        for name, v in out.items():
            a = v.detach().float().numpy()
            if a.ndim == 2 and a.shape[0] == N:
                a = a[rows]
            blob[f"{T.shape_key(shape)}:{name}"] = np.ascontiguousarray(a)
    path = os.path.normpath(os.path.join(TESTS, "golden", "submodules_reference.npz"))
    np.savez_compressed(path, **blob)
    print(f"{path}: {len(blob)} arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
