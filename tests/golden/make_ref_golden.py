#!/usr/bin/env python
"""Golden vectors from the REFERENCE's own model code.  Runs only where $CAPE_REFERENCE names its checkout.

`lib/models.py` of the reference is imported UNMODIFIED and executed on the TensorFlow-1 API shim of
oracle/tf1_shim.py (torch-CPU behind the ~70 TF symbols the file calls): `CAPE.build_graph(phase='train')` then runs
the reference's forward pass (condition nets, encoder, VAE sampling, decoder, discriminator on real and fake), its
`loss()` and its `training()` -- gradients, global-norm clip, momentum updates, including the quirks of
lib/models.py:466,470-472 -- on the fed batch.  The results go to tests/golden/ref_models_golden.npz:

  * x_hat, z_mean, z_logvar, the loss terms, the two learning rates;
  * per variable: the gradient the reference's optimiser saw (generator / condition nets: of loss_g; discriminator: of
    loss_d, which the reference computes and then discards) and the post-update value -- as l2 norm, sum and 64 sampled
    entries each, small tensors in full;
  * the variable inventory (names, shapes, creation order) the reference built;
  * the demo-phase graph (`build_graph(phase='demo')`): `op_decoder` on a given z_total and condition embeddings, the
    encoder's mean / log-variance, the condition embeddings -- what `decode` / `encode` / `encode_only_condition` run;
  * outputs of the reference's `base_model.chebyshev5 / b1leakyrelu / poolwT` on the inputs of tests/golden/inputs.py
    (BASELINE configs[0] among them): they pin the older ops_golden.npz, which came from a numpy transcription.

Inputs are the ones tests/parity.train_step uses (batch of 2 from cape_b200.synthetic.make_batch(seed 123), the
calibrated initial parameters, global_step 100), so the GPU parity tests, the oracle and this file meet on one update.
A second, smaller run covers the non-affine (GroupNorm) decoder of configs/CAPE_nz18_*.yaml at batch 1.

    CAPE_REFERENCE=/path/to/CAPE python tests/golden/make_ref_golden.py          (about a minute)
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
REF = os.environ.get("CAPE_REFERENCE", "")
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
if REF and REF not in sys.path:
    sys.path.append(REF)            # last: only `lib` (the reference's package) is meant to resolve there

OUT = os.path.join(HERE, "ref_models_golden.npz")
NSAMPLE = 64
OPS_STRIDE = 8


def reference_kwargs(cfg, h, batch_size, name="golden"):
    """The keyword arguments main.py:50-87 hands to models.CAPE, from our configuration dict."""
    return dict(L=h["L"], D=h["D"], U=h["U"], L_d=h["L_d"], D_d=h["D_d"], lr_scaler=cfg["lr_scaler"],
                lambda_gan=cfg["lambda_gan"], use_res_block=bool(cfg["use_res_block"]),
                use_res_block_dec=bool(cfg["use_res_block_dec"]), nz_cond2=cfg["nz_cond2"], cond2_dim=cfg["cond2_dim"],
                Kd=cfg["Kd"], n_layer_cond=cfg["n_layer_cond"], cond_encoder=bool(cfg["cond_encoder"]),
                reduce_dim=cfg["reduce_dim"], affine=bool(cfg["affine"]), lr_warmup=bool(cfg["lr_warmup"]),
                optim_condnet=bool(cfg["optim_condnet"]), F=list(cfg["F"]), K=list(cfg["K"]), p=h["p"], nz=cfg["nz"],
                loss=cfg["loss"], nn_input_channel=3, lr=cfg["lr"], decay_rate=cfg["decay_rate"],
                optimizer=cfg["optimizer"], decay_steps=cfg["decay_steps"], momentum=cfg["momentum"],
                cond_dim=cfg["cond_dim"], nz_cond=cfg["nz_cond"], regularization=cfg["regularization"],
                batch_size=batch_size, seed=cfg["seed"], lambda_recon=cfg["lambda_recon"],
                lambda_edge=cfg["lambda_edge"], lambda_latent=cfg["lambda_latent"], restart=True, name=name)


def run_reference(cfg, h, params, batch, step, momentum=None):
    """One `sess.run([op_train_g, op_train_d])` of the reference on the shim.  Returns a dict of numpy results.
    momentum: {variable name: accumulator} carried over from the previous update (None: zeros, a fresh optimiser)."""
    from oracle import tf1_shim as S
    from cape_b200 import topology as T
    S.install(template_vertices=T.template_mesh()[0])
    import contextlib
    import io
    N = batch["x_g"].shape[0]
    feeds = dict(data_g=batch["x_g"], data_d=batch["x_d"], condition_g=batch["cond_g"], condition2_g=batch["cond2_g"],
                 condition_d=batch["cond_d"], condition2_d=batch["cond2_d"], gt=batch["gt"], eps=batch["eps"])
    S.reset(feeds=feeds, params=params, global_step=step,
            slots={k + "/Momentum": v for k, v in (momentum or {}).items()})
    with contextlib.redirect_stdout(io.StringIO()):              # the reference prints its layer table
        from lib import models as RM                             # the reference's own module
        model = RM.CAPE(**reference_kwargs(cfg, h, N))
        model.build_graph(model.input_num_verts, model.nn_input_channel, phase="train")
    pre = {k: v.detach().clone().numpy() for k, v in S.VARS.items()}
    S.run_pending()
    n = lambda t: np.asarray(t.detach().as_subclass(torch.Tensor).numpy()) if isinstance(t, torch.Tensor) else np.asarray(t)
    out = dict(x_hat=n(model.op_prediction), z_mean=n(model.z_mean), z_logvar=n(model.z_logvar),
               recon=float(model.recon_loss), edge=float(model.edge_loss), latent=float(model.latent_loss),
               gan_g=float(model.loss_g), gan_d=float(model.loss_d), reg_g=float(model.fc_regularization_g),
               loss_g=float(model.op_loss_g), loss_d=float(model.op_loss_d), lr=np.asarray(S.RECORD["lr"], np.float64),
               global_step_after=int(S.GLOBAL_STEP))
    out["created"] = list(S.RECORD["created"])
    out["grads"] = {k: n(v) for k, v in S.RECORD["grads"].items() if v is not None}
    out["params_after"] = {k: n(v) for k, v in S.VARS.items()}
    out["params_before"] = pre
    out["momentum"] = {k[: -len("/Momentum")]: n(v) for k, v in S.RECORD["slots"].items() if k.endswith("/Momentum")}
    return out


def demo_feeds(cfg, N, seed=7):
    """Inputs of the demo-time ops (lib/models.py:323-347): a latent code, condition EMBEDDINGS, their concatenation."""
    rng = np.random.RandomState(seed)
    z = rng.normal(size=(N, cfg["nz"])).astype(np.float32)
    y = rng.normal(size=(N, cfg["nz_cond"])).astype(np.float32)
    y2 = rng.normal(size=(N, cfg["nz_cond2"])).astype(np.float32)
    return dict(z=z, cond_latent=y, cond2_latent=y2, z_total=np.concatenate([z, y, y2], 1))


def run_reference_demo(cfg, h, params, batch):
    """`build_graph(phase='demo')` of the reference on the shim: the ops its inference entry points run -- `op_decoder`
    (decode: z_total + condition embeddings -> vertices), `op_vae_mean / op_vae_var` (encode), the condition nets."""
    from oracle import tf1_shim as S
    from cape_b200 import topology as T
    S.install(template_vertices=T.template_mesh()[0])
    import contextlib
    import io
    N = batch["x_g"].shape[0]
    feeds = dict(data_g=batch["x_g"], data_d=batch["x_d"], condition_g=batch["cond_g"], condition2_g=batch["cond2_g"],
                 condition_d=batch["cond_d"], condition2_d=batch["cond2_d"], gt=batch["gt"], eps=batch["eps"])
    df = demo_feeds(cfg, N)
    feeds.update(df)
    S.reset(feeds=feeds, params=params, global_step=0)
    with contextlib.redirect_stdout(io.StringIO()):
        from lib import models as RM
        model = RM.CAPE(**reference_kwargs(cfg, h, N))
        model.build_graph(model.input_num_verts, model.nn_input_channel, phase="demo")
    n = lambda t: t.detach().as_subclass(torch.Tensor).numpy()
    return dict(decoded=n(model.op_decoder), vae_mean=n(model.op_vae_mean), vae_var=n(model.op_vae_var),
                cond_latent=n(model.op_cond_latent), cond2_latent=n(model.op_cond2_latent))


def run_reference_ops(h):
    """The reference's own `base_model.chebyshev5`, `b1leakyrelu` and `poolwT` (lib/models.py:69-152) on the inputs of
    tests/golden/inputs.py: BASELINE configs[0] (K = 6 conv on [1, 6890, 3]), conv + bias/leaky-ReLU + pool, un-pool."""
    from oracle import tf1_shim as S
    from cape_b200 import topology as T
    from inputs import golden_inputs
    S.install(template_vertices=T.template_mesh()[0])
    import contextlib
    import io
    g = golden_inputs()
    S.reset(params={"c1/weights": g["c1_W"], "cnp/weights": g["cnp_W"], "cnp/bias": g["cnp_b"].reshape(1, 1, -1)})
    with contextlib.redirect_stdout(io.StringIO()):
        from lib import models as RM
        m = RM.base_model(L=h["L"], D=h["D"], U=h["U"], F=[32], K=[2], p=h["p"], name="ops")
    tf = S.tf
    out = {}
    with tf.variable_scope("c1"):
        out["c1_y"] = m.chebyshev5(torch.from_numpy(g["c1_x"]), h["L"][0], 64, 6)
    with tf.variable_scope("cnp"):
        y = m.b1leakyrelu(m.chebyshev5(torch.from_numpy(g["cnp_x"]), h["L"][1], 32, 2))
        out["cnp_y"] = m.poolwT(y, h["D"][1])
    out["up_y"] = m.poolwT(torch.from_numpy(g["up_x"]), h["U"][1])
    return {k: v.detach().as_subclass(torch.Tensor).numpy() for k, v in out.items()}


def sample_index(name, size):
    """The same 64 positions of a tensor in the generator and in the test (seeded by the variable name)."""
    seed = int.from_bytes(name.encode()[-4:].rjust(4, b"\0"), "little") ^ (size & 0x7fffffff)
    return np.random.RandomState(seed % (2 ** 31)).randint(0, size, size=min(NSAMPLE, size))


def pack(tag, res, store):
    for k in ("x_hat", "z_mean", "z_logvar", "lr"):
        store["%s/%s" % (tag, k)] = np.asarray(res[k])
    for k in ("recon", "edge", "latent", "gan_g", "gan_d", "reg_g", "loss_g", "loss_d", "global_step_after"):
        store["%s/%s" % (tag, k)] = np.asarray(res[k], np.float64)
    store["%s/var_names" % tag] = np.asarray([c[0] for c in res["created"]])
    store["%s/var_shapes" % tag] = np.asarray([",".join(map(str, c[1])) for c in res["created"]])
    for kind in ("grads", "params_after"):
        for name, v in res[kind].items():
            v = np.asarray(v, np.float32)
            base = "%s/%s/%s" % (tag, kind, name)
            store[base + "#l2"] = np.asarray(np.sqrt((v.astype(np.float64) ** 2).sum()))
            store[base + "#sum"] = np.asarray(v.astype(np.float64).sum())
            flat = v.reshape(-1)
            if flat.size <= 4096:
                store[base + "#full"] = v
            else:
                store[base + "#sample"] = flat[sample_index(name, flat.size)]


def configs():
    from cape_b200.params import NZ18_PLAIN, NZ64_AFFINE
    return (("nz64", dict(NZ64_AFFINE, decay_steps=10), 2, 100), ("nz18", dict(NZ18_PLAIN, decay_steps=10), 1, 100))


def inputs(cfg, h, N, seed=123):
    import parity
    from cape_b200.params import param_specs
    from cape_b200.synthetic import make_batch
    specs = param_specs(cfg, [l.shape[0] for l in h["L"]], [l.shape[0] for l in h["L_d"]])
    return parity.calibrated_params(specs, seed, 0.05), make_batch(N, cfg["nz"], seed=seed)


def four_layer_case(h):
    """(tag, cfg, hierarchy) of the 4-conv-layer variant: F = [nf, 2nf, 2nf, nf], ds_factors [1, 2, 1, 1]."""
    from cape_b200 import main as M
    from cape_b200.params import NZ64_AFFINE
    L, D, U, p = M.build_hierarchy(num_conv_layers=4, ds_factor=2)
    cfg = dict(NZ64_AFFINE, F=[64, 128, 128, 64], K=[2] * 4, decay_steps=10)
    return "nz64_l4", cfg, dict(L=L, D=D, U=U, p=p, L_d=h["L_d"], D_d=h["D_d"])


def second_batch(cfg, N, seed=123):
    from cape_b200.synthetic import make_batch
    return make_batch(N, cfg["nz"], seed=seed + 1000)            # the batch tests/parity.train_step draws for update 2


def main():
    from cape_b200 import topology as T
    L, D, U, p, L_d, D_d, _ = T.load_graph_mtx(load_for_demo=True)
    h = dict(L=L, D=D, U=U, p=p, L_d=L_d, D_d=D_d)
    store = {}
    for tag, cfg, N, step in configs():
        params, batch = inputs(cfg, h, N)
        res = run_reference(cfg, h, params, batch, step)
        print("%s: x_hat %s  recon %.6f edge %.6f latent %.6f gan_g %.6f gan_d %.6f  lr %s  step -> %d  (%d variables)"
              % (tag, res["x_hat"].shape, res["recon"], res["edge"], res["latent"], res["gan_g"], res["gan_d"], res["lr"],
                 res["global_step_after"], len(res["created"])))
        pack(tag, res, store)
        if tag == "nz64":
            # a SECOND update on top of the first: momentum accumulators, the shared global_step (now 102) and the
            # updated parameters carried over, a fresh batch -- what two consecutive sess.run calls of fit() do
            batch2 = second_batch(cfg, N)
            res2 = run_reference(cfg, h, res["params_after"], batch2, res["global_step_after"], momentum=res["momentum"])
            print("%s_u2: recon %.6f gan_d %.6f lr %s step -> %d" % (tag, res2["recon"], res2["gan_d"], res2["lr"],
                                                                    res2["global_step_after"]))
            pack(tag + "_u2", res2, store)
    tag, cfg, N, step = configs()[0]
    params, batch = inputs(cfg, h, N)
    for k, v in run_reference_demo(cfg, h, params, batch).items():
        store["%s/demo/%s" % (tag, k)] = v
    # --num_conv_layers 4 (main.py:31-32,56-57) on the hierarchy cape_b200.mesh_sampling generates from the template:
    # variable inventory, forward outputs and losses of the reference on an architecture it ships no fixtures for
    tag4, cfg4, h4 = four_layer_case(h)
    params4, batch4 = inputs(cfg4, h4, 1)
    res4 = run_reference(cfg4, h4, params4, batch4, 100)
    print("%s: recon %.6f gan_d %.6f (%d variables)" % (tag4, res4["recon"], res4["gan_d"], len(res4["created"])))
    store[tag4 + "/var_names"] = np.asarray([c[0] for c in res4["created"]])
    store[tag4 + "/var_shapes"] = np.asarray([",".join(map(str, c[1])) for c in res4["created"]])
    store[tag4 + "/x_hat"] = res4["x_hat"]
    for k in ("recon", "edge", "latent", "gan_g", "gan_d"):
        store["%s/%s" % (tag4, k)] = np.asarray(res4[k], np.float64)
    ops = run_reference_ops(h)
    prev = np.load(os.path.join(HERE, "ops_golden.npz"))
    for k, v in ops.items():
        store["ops/" + k] = v.astype(np.float32).reshape(-1)[::OPS_STRIDE]         # every 8th element keeps the file small
        print("ops %s: reference vs the committed known answer (numpy transcription): max rel %.2e"
              % (k, np.abs(v - prev[k]).max() / np.abs(prev[k]).max()))
    np.savez_compressed(OUT, **store)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
