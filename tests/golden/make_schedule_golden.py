"""Generates tests/golden/hf_polynomial_warmup.npz: the learning rate of every step of transformers' torch twin of HF
`WarmUp` + Keras `PolynomialDecay` (`get_polynomial_decay_schedule_with_warmup(lr_end=1e-7, power=1.0)`, warm-up over
10 % of the steps as polus/schedulers.py:5-23) for the cases tests/test_host_cpu.py checks.
Needs torch + transformers (CPU only):  python tests/golden/make_schedule_golden.py"""
import os

import numpy as np
import torch
from transformers.optimization import get_polynomial_decay_schedule_with_warmup

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = ((200, 3e-4), (1000, 5e-5), (37, 1e-3))   # (training steps, peak learning rate)


def main():
    out = {"n_steps": np.asarray([n for n, _ in CASES], np.int64), "lr": np.asarray([lr for _, lr in CASES], np.float64)}
    for i, (n_steps, lr) in enumerate(CASES):
        opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=lr)
        hf = get_polynomial_decay_schedule_with_warmup(opt, num_warmup_steps=int(n_steps * 0.1), num_training_steps=n_steps,
                                                       lr_end=1e-7, power=1.0)
        lrs = []
        for _ in range(n_steps + 1):
            lrs.append(hf.get_last_lr()[0])
            opt.step()
            hf.step()
        out[f"lrs_{i}"] = np.asarray(lrs, np.float64)   # lrs_i[step], steps 0 .. n_steps
    np.savez_compressed(os.path.join(HERE, "hf_polynomial_warmup.npz"), **out)
    print("wrote hf_polynomial_warmup.npz:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
