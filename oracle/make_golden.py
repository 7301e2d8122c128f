"""TEST INFRASTRUCTURE -- generate tests/golden/*.npz from the UNMODIFIED reference module.

Needs an unmodified CFDBench `src/` tree: CFDBENCH_SRC, else oracle/build_ref.py's default location:

    CFDBENCH_SRC=/path/to/CFDBench/src PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden.py

For each case it (1) builds the reference `Fno2d` (reference src/models/fno/fno2d.py:115) with
weights from `cfdbench_b200.synth.make_state_dict(seed)` loaded through `load_state_dict`,
(2) runs forward / loss / backward / generate_many on CPU fp32, (3) checks that both oracles
(`oracle/fno_torch_port.py`, `oracle/fno_numpy.py`) reproduce it, and (4) stores seeds + inputs +
reference outputs.  Weights are NOT stored (tests regenerate them from the seed).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import build_ref  # noqa: E402

sys.path.insert(0, build_ref.source_dir())
sys.dont_write_bytecode = True

from models.fno.fno2d import Fno2d, SpectralConv2d_fast  # noqa: E402  (the reference)
from models.loss import loss_name_to_fn  # noqa: E402

from cfdbench_b200 import synth  # noqa: E402
from oracle import fno_numpy as onp  # noqa: E402
from oracle import fno_torch_port as opt  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")

CASES = [
    # name, problem, batch, weight seed, batch seed, spectral gain, rollout steps, spectral weight gradients stored
    ("cavity_b2_gain200", "cavity", 2, 101, 201, 200.0, 3, False),
    ("cylinder_b2_gain200", "cylinder", 2, 102, 202, 200.0, 3, True),
    ("cavity_b1_default_init", "cavity", 1, 103, 203, 1.0, 20, False),
]
# hidden activations are stored for these channels only, which keeps every fixture under 1 MB
ACT_CHANNELS = np.arange(0, synth.HIDDEN, 8)


def ref_model(sd: dict, p: int) -> Fno2d:
    m = Fno2d(in_chan=2, out_chan=2, n_case_params=p, loss_fn=loss_name_to_fn("nmse"),
              num_layers=synth.DEPTH, hidden_dim=synth.HIDDEN, modes1=synth.MODES, modes2=synth.MODES)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return m


def main() -> None:
    torch.set_num_threads(8)
    os.makedirs(GOLD, exist_ok=True)
    for name, problem, b, wseed, bseed, gain, steps, spectral_grads in CASES:
        p = synth.n_case_params(problem)
        sd = synth.make_state_dict(wseed, n_params=p, spectral_gain=gain)
        batch = synth.make_batch(bseed, b, problem)
        tb = {k: torch.from_numpy(v) for k, v in batch.items()}
        model = ref_model(sd, p)

        # hooks: lift output and every block output
        acts = []
        hooks = [model.fc0.register_forward_hook(lambda m, i, o: acts.append(o.detach().numpy().copy()))]
        for blk in model.blocks:
            hooks.append(blk.register_forward_hook(lambda m, i, o: acts.append(o.detach().numpy().copy())))
        out = model(**tb)
        for hk in hooks:
            hk.remove()
        out["loss"]["nmse"].backward()
        grads = {k: v.grad.numpy().copy() for k, v in model.named_parameters()}
        with torch.no_grad():
            roll = model.generate_many(tb["inputs"], tb["case_params"], tb["mask"], steps)
            spec = model.blocks[0].conv0(torch.from_numpy(acts[0])).numpy()

        # --- pin the oracles against the reference ------------------------------------------
        pp = opt.params_from_numpy(sd, requires_grad=True)
        pout = opt.forward(pp, tb["inputs"], tb["case_params"], tb["mask"], tb["label"], return_acts=True)
        assert torch.equal(pout["preds"], out["preds"]), "torch port is not bit-identical to the reference"
        for k in out["loss"]:
            assert torch.equal(pout["loss"][k], out["loss"][k]), k
        pout["loss"]["nmse"].backward()
        for k, g in grads.items():
            assert np.array_equal(pp[k].grad.numpy(), g), f"port grad {k}"
        proll = opt.rollout(opt.params_from_numpy(sd), tb["inputs"], tb["case_params"], tb["mask"], steps)
        for a, r in zip(proll, roll):
            assert torch.equal(a, r)

        nout = onp.fno_forward(sd, batch["inputs"], batch["case_params"], batch["mask"], batch["label"],
                               return_acts=True)
        e = onp.rel_l2(out["preds"].detach().numpy(), nout["preds"])
        assert e < 2e-6, f"numpy oracle vs reference preds rel-L2 {e}"
        for i, a in enumerate(acts):
            ea = onp.rel_l2(a, nout["acts"][i])
            assert ea < 2e-6, (i, ea)
        ngr = onp.fno_backward(sd, batch["inputs"], batch["case_params"], batch["mask"], batch["label"])
        worst = 0.0
        for k, g in grads.items():
            eg = np.linalg.norm(g - ngr[k]) / np.linalg.norm(ngr[k])
            worst = max(worst, eg)
            assert eg < 5e-5, f"numpy oracle grad {k}: {eg}"
        es = onp.rel_l2(spec, onp.spectral_conv(acts[0], sd["blocks.0.conv0.weights1"],
                                                sd["blocks.0.conv0.weights2"]))
        assert es < 2e-6, es
        print(f"{name}: numpy-vs-ref preds {e:.2e}, spectral {es:.2e}, worst grad {worst:.2e}; port bit-exact")

        # --- store ------------------------------------------------------------------------------
        store = dict(
            problem=np.array(problem), weight_seed=np.array(wseed), batch_seed=np.array(bseed),
            spectral_gain=np.array(gain), steps=np.array(steps),
            preds=out["preds"].detach().numpy(),
            loss=np.array([out["loss"][k].item() for k in ("mse", "rmse", "mae", "nmse")], dtype=np.float64),
            rollout=np.stack([r.numpy() for r in roll]),
            act_channels=ACT_CHANNELS,
            act0_b0=acts[0][:1, ACT_CHANNELS], act1_b0=acts[1][:1, ACT_CHANNELS], act4_b0=acts[-1][:1, ACT_CHANNELS],
            spectral0_b0=spec[:1, ACT_CHANNELS],
        )
        for k in ("fc0.weight", "fc0.bias", "fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias",
                  "blocks.0.w0.weight", "blocks.0.w0.bias", "blocks.3.w0.weight", "blocks.3.w0.bias"):
            store["grad::" + k] = grads[k]
        for k in ("blocks.0.conv0.weights1", "blocks.0.conv0.weights2", "blocks.3.conv0.weights1",
                  "blocks.3.conv0.weights2") if spectral_grads else ():
            store["gradslice::" + k] = grads[k][:, :, ::4, ::4]           # (32,32,3,3) complex
            store["gradnorm::" + k] = np.array(np.linalg.norm(grads[k]))
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **store)

    # layer-level known-answer fixture straight from SpectralConv2d_fast with non-default sizes is
    # not needed: the CUDA path is specialised on (64,64,32,12,12) like the reference's config.
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
