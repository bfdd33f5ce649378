"""Golden gradients of the PPO update, produced by the REAL reference update on CPU (the setup of gen_ppo_golden.py:
hidden 32, 2 episodes x 36 steps x 4 envs, K_epochs 2, minibatches of 36 steps in the recorded sampler order).

ppo_golden.npz pins the parameters after four Adam steps, and Adam's step hardly depends on a gradient's scale.  This
fixture pins the gradients themselves: at every `step()` of the three optimisers it records every parameter's `.grad`
(`step{k}/{job,mch,crit}/<key>`, k = 0..3 in call order), and for the global critic also the gradient before
`clip_grad_norm_` (`step{k}/crit_preclip/<key>`).  Minibatch 0 starts from the seeded weights, so its gradients can
be recomputed without replaying any optimiser state.

Run in the build container only:  python tests/golden/gen_ppo_grad_golden.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import gen_ppo_golden as gpg  # noqa: E402


def main():
    rec = {}
    counts = {"job": 0, "mch": 0, "crit": 0}
    names = {}

    def grads(tag, net):
        return {"%s/%s" % (tag, k): p.grad.detach().numpy().astype(np.float32).copy()
                for k, p in net.named_parameters() if p.grad is not None}

    def wrap_step(opt, tag, net):
        step = opt.step

        def recorded(*a, **k):
            rec.update({"step%d/%s" % (counts[tag], n): v for n, v in grads(tag, net).items()})
            counts[tag] += 1
            return step(*a, **k)
        opt.step = recorded

    clip = torch.nn.utils.clip_grad_norm_

    def recorded_clip(params, *a, **k):
        params = list(params)
        net = names.get(tuple(id(p) for p in params))
        if net is not None and any(p.grad is not None for p in params):
            # the reference clips the actors before their backward (no gradient yet); only the critic's call sees one
            rec.update({"step%d/crit_preclip/%s" % (counts["crit"], n.split("/", 1)[1]): v
                        for n, v in grads("crit", net).items()})
        return clip(params, *a, **k)

    def before_update(ppo):
        wrap_step(ppo.job_actor_optimizer, "job", ppo.job_actor)
        wrap_step(ppo.machine_actor_optimizer_gcn, "mch", ppo.machine_actor_gcn)
        wrap_step(ppo.global_critic_optimizer, "crit", ppo.global_critic)
        names[tuple(id(p) for p in ppo.global_critic.parameters())] = ppo.global_critic
        torch.nn.utils.clip_grad_norm_ = recorded_clip

    try:
        out, _ = gpg.run_update(before_update)
    finally:
        torch.nn.utils.clip_grad_norm_ = clip
    assert counts["job"] == counts["mch"] == counts["crit"] == 2 * out["K_epochs"]
    assert all("step%d/crit_preclip/critic.linears.0.weight" % k in rec for k in range(counts["crit"]))
    rec["H"], rec["mini_bs"], rec["orders"] = out["H"], out["mini_bs"], out["orders"]
    np.savez_compressed(os.path.join(HERE, "ppo_grad_golden.npz"), **rec)
    print("wrote ppo_grad_golden.npz: %d arrays, %d KB" % (len(rec), os.path.getsize(os.path.join(HERE, "ppo_grad_golden.npz")) // 1024))


if __name__ == "__main__":
    main()
