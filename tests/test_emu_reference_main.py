"""The reference's caller driving the drop-in (VERDICT r1 #9, SURVEY 8b): `from Models import MMSSL, Discriminator` (main.py:27)
resolves to mmssl_b200/Models.py, and the reference's `Trainer` runs three iterations of its batch loop on the cuemu device --
seeded construction, both torch optimisers, no-grad forward, Discriminator step with gradient penalty, forward with grad,
losses on our outputs indexed with Python lists, backward through MMSSLForwardFn, AdamW on our parameters -- and must
reproduce what the UNMODIFIED reference trainer recorded with the reference's model (tests/golden/gan_trace.npz, minted by
tests/golden/make_golden_gan.py: every random draw injected, gradients before and parameters after each optimiser step of
all three iterations).

The original sources are not part of this repository, so the caller is restated in `_ReferenceCaller` below: construction
(main.py:54-80), weights_init (main.py:135-138) and the batch loop (main.py:333-431), with the loss and GAN pieces of the
oracle (oracle/mmssl_oracle.py, oracle/gan_oracle.py; both pinned to the reference by their own golden tests) and torch
autograd and optimisers for everything else, as in the reference."""
import importlib.util
import json
import os
import random
import sys

import numpy as np
import scipy.sparse as sp
import torch
import torch.nn as nn
from torch import autograd, optim

from oracle import gan_oracle as GO, mmssl_oracle as O
from tests.cuemu import harness
from tests.golden_util import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LIVE = ["image_trans.weight", "image_trans.bias", "text_trans.weight", "text_trans.bias", "user_id_embedding.weight",
        "item_id_embedding.weight", "weight_dict.w_self_attention_cat"]


class _Replay(nn.Module):
    """nn.Dropout stand-in that multiplies by the masks the reference run drew (in the order it drew them)."""

    def __init__(self, masks):
        super().__init__()
        self.masks, self.i = masks, 0

    def forward(self, x):
        if not self.training:
            return x
        m = torch.from_numpy(self.masks[self.i])
        self.i += 1
        return x * m


class _ReferenceCaller:
    """What the reference's Trainer does around `MMSSL` and `Discriminator`, for the recorded run (T = 1, batch size B)."""

    def __init__(self, z, c, seed):
        from Models import Discriminator, MMSSL
        self.c = c
        self.R = sp.csr_matrix((np.ones(len(z["train_rows"]), np.float32), (z["train_rows"], z["train_cols"])),
                               shape=(c["U"], c["I"]))
        ui, iu = O.build_graphs(self.R)
        self.graphs = [ui, iu, ui, iu, ui, iu]             # modality graphs alias ui / iu at the start (main.py:68-69)
        self.cfg = O.HotPathConfig(embed_size=c["d"], n_layers=c["n_layers"], head_num=c["head_num"], id_cat_rate=c["id_cat_rate"],
                                   model_cat_rate=c["model_cat_rate"], drop_rate=c["drop_rate"], tau=c["tau"], cl_rate=c["cl_rate"],
                                   emb_decay=c["emb_decay"], feat_reg_decay=c["feat_reg_decay"], batch_size=c["B"])
        self.gcfg = GO.GanConfig(G_drop1=c["G_drop1"], G_drop2=c["G_drop2"], gp_rate=c["gp_rate"], G_rate=c["G_rate"], D_lr=c["D_lr"],
                                 log_log_scale=c["log_log_scale"], real_data_tau=c["real_data_tau"], ui_pre_scale=c["ui_pre_scale"],
                                 m_topk_rate=c["m_topk_rate"], T=c["T"])
        np.random.seed(seed); random.seed(seed); torch.manual_seed(seed)
        self.model = MMSSL(c["U"], c["I"], c["d"], [c["d"]] * c["n_layers"], [0.1] * c["n_layers"], z["image_feats"], z["text_feats"]).cuda()
        self.D = Discriminator(c["I"]).cuda()
        for m in self.D.modules():                         # weights_init
            if isinstance(m, nn.Linear):
                nn.init.kaiming_normal_(m.weight)
                m.bias.data.fill_(0)
        self.optim_D = optim.Adam(self.D.parameters(), lr=c["D_lr"], betas=(0.5, 0.9))
        self.optimizer_D = optim.AdamW([{"params": self.model.parameters()}], lr=c["lr"])
        self.index = {"image": ([], []), "text": ([], [])}

    def u_sim(self, users, uf, itf):
        return GO.u_sim(users, uf, itf, self.R, self.c["B"])

    def step(self, idx, users, pos, neg, gumbel_u, alpha):
        g, D = self.gcfg, self.D
        self.model.train()
        with torch.no_grad():
            outs = self.model(*self.graphs)
        ui_sim = self.u_sim(users, outs[0], outs[1]).detach()
        inputf = torch.cat((self.u_sim(users, outs[4], outs[2]).detach(), self.u_sim(users, outs[5], outs[3]).detach()), dim=0)
        lossf = D(inputf).mean()
        inputr = GO.real_rows(users, self.R, gumbel_u, ui_sim, g)
        inputr = torch.cat((inputr, inputr), dim=0)
        lossr = -D(inputr).mean()
        a = alpha.expand_as(inputr)                        # gradient penalty (main.py:140-160)
        inter = (a * inputr + (1 - a) * inputf.detach()).requires_grad_(True)
        out = D(inter)
        gi = autograd.grad(outputs=out, inputs=inter, grad_outputs=torch.ones_like(out), create_graph=True, retain_graph=True,
                           only_inputs=True)[0]
        gp = ((gi.norm(2, dim=1) - 1) ** 2).mean() * g.gp_lambda
        loss_D = lossr + lossf + g.gp_rate * gp
        self.optim_D.zero_grad()
        loss_D.backward()
        self.optim_D.step()

        outs = self.model(*self.graphs)
        hot, _ = O.hot_loss(outs, users, pos, neg, self.c["I"], self.cfg, literal=True)
        g_img, g_txt = self.u_sim(users, outs[4], outs[2]), self.u_sim(users, outs[5], outs[3])
        if idx % g.T == 0 and idx != 0:                    # modality graphs rebuilt from the collected top-k pairs
            gi_ui, gi_iu = GO.rebuild_graphs(*self.index["image"], self.c["U"], self.c["I"])
            gt_ui, gt_iu = GO.rebuild_graphs(*self.index["text"], self.c["U"], self.c["I"])
            self.graphs = self.graphs[:2] + [gi_ui, gi_iu, gt_ui, gt_iu]
            self.index = {"image": ([], []), "text": ([], [])}
        else:
            for key, sim in (("image", g_img), ("text", g_txt)):
                x, y = GO.topk_pairs(users, sim, self.c["I"], g)
                self.index[key][0].extend(x); self.index[key][1].extend(y)
        G_lossf = -D(torch.cat((g_img, g_txt), dim=0)).mean()
        batch_loss = hot + g.G_rate * G_lossf
        self.optimizer_D.zero_grad()
        batch_loss.backward()
        self.optimizer_D.step()


def test_reference_trainer_runs_on_the_drop_in_and_reproduces_its_own_trace(monkeypatch):
    monkeypatch.syspath_prepend(os.path.join(ROOT, "tests", "golden"))
    from make_golden_gan import CASE
    z = np.load(os.path.join(ROOT, "tests", "golden", "gan_trace.npz"))
    cfg = json.loads(str(z["cfg"]))
    harness.set_order("fwd")
    harness.emulated_device(monkeypatch)
    monkeypatch.setattr(nn.Module, "cuda", lambda self, *a, **k: self)
    # the drop-in file under the name the reference imports
    spec = importlib.util.spec_from_file_location("Models", os.path.join(ROOT, "mmssl_b200", "Models.py"))
    dropin = importlib.util.module_from_spec(spec)
    monkeypatch.setitem(sys.modules, "Models", dropin)
    spec.loader.exec_module(dropin)

    tr = _ReferenceCaller(z, cfg, CASE["seed"])
    named = dict(tr.model.named_parameters())
    # seeded construction draws the reference's initial values (parameter creation order, Models.py:28-66) ...
    for k in LIVE:
        assert torch.equal(named[k].detach(), torch.from_numpy(z["G0/" + k])), k
    for k, v in tr.D.state_dict().items():
        assert torch.equal(v, torch.from_numpy(z["D0/" + k])), k
    # ... every random draw of the recorded run is replayed
    tr.model.dropout = _Replay(z["mask_model"])
    tr.D.net[3], tr.D.net[7] = _Replay(z["mask_d1"]), _Replay(z["mask_d2"])

    got = {"Ggrad": [], "Gparam": [], "Dstate": []}
    tr.optimizer_D.register_step_pre_hook(lambda o, a, k: got["Ggrad"].append({n: named[n].grad.detach().clone() for n in LIVE}))
    tr.optimizer_D.register_step_post_hook(lambda o, a, k: got["Gparam"].append({n: named[n].detach().clone() for n in LIVE}))
    tr.optim_D.register_step_post_hook(lambda o, a, k: got["Dstate"].append({n: v.detach().clone() for n, v in tr.D.state_dict().items()}))
    for s in range(cfg["steps"]):
        users, pos, neg = ([int(v) for v in z["sample"][s][j]] for j in range(3))      # Python lists, like the reference's sampler
        tr.step(s, users, pos, neg, torch.from_numpy(z["gumbel_u"][s]), torch.from_numpy(z["alpha"][s]))

    assert len(got["Gparam"]) == cfg["steps"] and tr.model.dropout.i == len(z["mask_model"]) and tr.D.net[3].i == len(z["mask_d1"])
    for s in range(cfg["steps"]):
        for k in LIVE:
            e = rel_err(got["Ggrad"][s][k], torch.from_numpy(z["Ggrad/" + k][s]))
            assert e < 1e-4, (s, "Ggrad", k, e)
            e = rel_err(got["Gparam"][s][k], torch.from_numpy(z["Gparam/" + k][s]))
            assert e < 1e-4, (s, "Gparam", k, e)
        for k in cfg["d_state_names"]:
            # biases in front of a BatchNorm have an exactly-zero gradient in exact arithmetic: what Adam normalises there is
            # rounding noise of the reference's own torch ops (tests/fullstep_check.py treats them the same way)
            # (and the running means of those BatchNorms follow the noise-driven biases from the second iteration on)
            if "num_batches_tracked" in k or k in ("net.0.bias", "net.4.bias") or (s > 0 and k.endswith("running_mean")):
                continue
            # the Discriminator is the reference's own torch module on both sides; it sees our outputs (1e-6 away from the
            # reference's) and Adam on its scalar output bias shows 1.1e-4 after three iterations: 1e-3 for this bystander
            e = rel_err(got["Dstate"][s][k], torch.from_numpy(z["Dstate/" + k][s]))
            assert e < 1e-3, (s, "Dstate", k, e)
