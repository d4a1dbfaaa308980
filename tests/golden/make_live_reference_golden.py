"""Golden vectors for the tests that compare with the unmodified reference `Mapper` run beside our code
(tests/test_oracle.py, tests/test_parity_gpu.py).  The reference is loaded through oracle/build_ref.py and runs on the
CPU; the tests then need only this file.  Large outputs are stored as a fixed row sample; the reference's initial
mapping (its seeded float64 draw cast to float32) is stored as a sha256 of its bytes.

    python tests/golden/make_live_reference_golden.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import build_ref  # noqa: E402
from oracle.tangram_oracle import synthetic_inputs  # noqa: E402
from tests.helpers import sha256_f32  # noqa: E402

ref = build_ref.load()
torch.set_num_threads(1)


def sample_rows(n, k, seed):
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def losses(hist, key):
    return np.array([float(x) for x in hist[key]], dtype=np.float64)


# test_oracle_matches_live_reference_autograd: loss and dL/dM of the first epoch
inp = synthetic_inputs(500, 130, 70, seed=9)
r = ref.Mapper(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, lambda_g2=0.2, lambda_r=1e-4, random_state=5)
M0 = r.M.detach().numpy().copy()
loss = r._loss_fn(verbose=False)[0]
loss.backward()
rows = sample_rows(500, 128, 0)
np.savez_compressed(os.path.join(HERE, "live_reference_autograd.npz"), M0_sha256=np.array(sha256_f32(M0)), total_loss=np.array(float(loss.detach())),
                    rows=rows, grad_rows=r.M.grad.numpy()[rows])

# test_second_train_call_restarts_adam_like_the_reference: train(4) then train(3) on the same Mapper
inp = synthetic_inputs(60, 25, 12, seed=4)
r = ref.Mapper(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, random_state=7, device="cpu")
r.train(4, print_each=None)
out, hist = r.train(3, print_each=None)
np.savez_compressed(os.path.join(HERE, "live_reference_second_train.npz"), output=out, total_loss=losses(hist, "total_loss"))

# test_live_reference_on_the_same_gpu: 30 epochs from the reference's own seed-42 draw
inp = synthetic_inputs(3000, 700, 300, seed=31)
r = ref.Mapper(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, random_state=42, device="cpu")
M0 = r.M.detach().numpy().copy()
out, hist = r.train(num_epochs=30, learning_rate=0.1, print_each=None)
rows = sample_rows(3000, 32, 0)
np.savez_compressed(os.path.join(HERE, "live_reference_30_epochs.npz"), M0_sha256=np.array(sha256_f32(M0)), total_loss=losses(hist, "total_loss"),
                    main_loss=losses(hist, "main_loss"), rows=rows, out_rows=out[rows])
for f in sorted(os.listdir(HERE)):
    if f.startswith("live_reference_"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
