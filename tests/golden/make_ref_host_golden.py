#!/usr/bin/env python
"""Golden data of the REFERENCE's host-side code: what tests/test_config.py and tests/test_reference_golden.py compare
this package with, recorded once from a checkout of the reference so that those tests run without it.

  * ref_config_golden.json: the reference's shipped yaml files (configs/*.yaml), the flag table its own
    `parse_config` declares (config_parser.py:11-63, recorded with a stand-in for `configargparse`) and the parameters
    of its `models.CAPE` constructor chain;
  * ref_host_golden.npz: the reference's `load_data.BodyData` on seeded files, the meshes its `demos.demo_simple`
    writes, the batches its `CAPE.fit` feeds, the results of its `predict` / `evaluate` / `encode` /
    `encode_only_condition` / `decode` loops (all driven by the deterministic stand-ins the tests define) and the
    learning rates of its `training()`.  Arrays larger than a few hundred kB are stored as a seeded sample
    (`test_reference_golden.sample_index`) plus their float64 sum.

    CAPE_REFERENCE=/path/to/CAPE python tests/golden/make_ref_host_golden.py
"""
import contextlib
import inspect
import io
import json
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)

import make_ref_golden as G  # noqa: E402  (puts the reference's checkout on sys.path)
import test_reference_golden as TR  # noqa: E402  (the stand-ins and seeded inputs both sides share)

OUT_JSON = os.path.join(HERE, "ref_config_golden.json")
OUT_NPZ = os.path.join(HERE, "ref_host_golden.npz")


def store_sampled(store, name, a):
    a = np.asarray(a)
    store[name + "#sample"] = a.reshape(-1)[TR.sample_index(name, a.size)]
    store[name + "#sum"] = np.asarray(a, np.float64).sum()
    store[name + "#shape"] = np.asarray(a.shape, np.int64)


@contextlib.contextmanager
def _stubs():
    saved = {k: sys.modules.get(k) for k in TR.STUBBED}
    try:
        yield
    finally:
        from oracle import tf1_shim as S
        S.SESSION_FACTORY = None
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def reference_config():
    """The reference's yaml files, its parse_config flag table and its constructor's parameters."""
    import argparse
    import importlib.util
    cfg_dir = os.path.join(G.REF, "configs")
    configs = {fn: open(os.path.join(cfg_dir, fn)).read() for fn in sorted(os.listdir(cfg_dir))}
    recorded = []

    class ArgParser(object):
        def __init__(self, *a, **k):
            pass

        def add_argument(self, flag, **kw):
            recorded.append((flag.lstrip("-"), kw))

        def parse_known_args(self, *a, **k):
            return argparse.Namespace(**{n: kw.get("default") for n, kw in recorded}), []

    stub = types.ModuleType("configargparse")
    stub.ArgParser, stub.ArgumentDefaultsHelpFormatter, stub.DefaultConfigFileParser = ArgParser, object, object
    saved = sys.modules.get("configargparse")
    sys.modules["configargparse"] = stub
    try:
        spec = importlib.util.spec_from_file_location("ref_config_parser", os.path.join(G.REF, "config_parser.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.parse_config()
    finally:
        if saved is None:
            sys.modules.pop("configargparse")
        else:
            sys.modules["configargparse"] = saved
    flags = [[n, kw.get("type", str).__name__, kw.get("default"),
              None if kw.get("choices") is None else list(kw["choices"])] for n, kw in recorded[1:]]
    config_flag = dict(name=recorded[0][0], is_config_file=bool(recorded[0][1].get("is_config_file")),
                       default=recorded[0][1].get("default"))
    with _stubs():
        from oracle import tf1_shim as S
        S.install(template_vertices=np.zeros((6890, 3)))
        from lib import models as RM
        chain = [c for c in RM.CAPE.__mro__ if "__init__" in vars(c) and c is not object]
    # CAPE.__init__ hands **kwargs to base_model.__init__: the named parameters of the whole chain, in order
    ctor = []
    for c in chain:
        for n, prm in inspect.signature(c.__init__).parameters.items():
            if prm.kind is prm.VAR_KEYWORD:
                assert c is not chain[-1], "the last constructor of the chain takes any keyword"
            elif n != "self" and n not in [x[0] for x in ctor]:
                ctor.append([n, prm.default is inspect.Parameter.empty])
    return dict(configs=configs, flags=flags, config_flag=config_flag, ctor_params=ctor)


def reference_body_data(store, tmp):
    from oracle import tf1_shim as S
    with _stubs():
        S.install()
        from lib import load_data as RL
        with contextlib.redirect_stdout(io.StringIO()):
            ref = RL.BodyData(reference_mesh_file="unused.obj", **TR.body_data_files(tmp))
    for k in TR.BODY_DATA_KEYS:
        store["body_data/" + k] = getattr(ref, k)
    store["body_data/n_vertex"] = np.asarray(ref.n_vertex)


def reference_demo_simple(store, tmp):
    import importlib.util
    from cape_b200 import demos as ours
    from cape_b200 import topology
    from oracle import tf1_shim as S
    with _stubs():
        S.install()
        v, f = topology.template_mesh()

        class _Tri(object):
            def __init__(self, vertices=None, faces=None):
                self.vertices, self.faces = vertices, faces

            def export(self, path):
                ours.write_obj(path, self.vertices, self.faces)

        sys.modules["trimesh"] = types.ModuleType("trimesh")
        sys.modules["trimesh"].load = lambda *a, **k: _Tri(np.asarray(v), np.asarray(f))
        sys.modules["trimesh"].Trimesh = _Tri
        scratch = os.path.join(tmp, "ref")
        os.mkdir(scratch)
        os.symlink(os.path.join(G.REF, "data"), os.path.join(scratch, "data"))
        spec = importlib.util.spec_from_file_location("ref_demos", os.path.join(G.REF, "demos.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.__file__ = os.path.join(scratch, "demos.py")
        with contextlib.redirect_stdout(io.StringIO()):
            ref = mod.demo_simple(TR._FakeModel(), "x", 123)
            ref.sample_vary_clotype()
    files = sorted(os.listdir(ref.results_dir))
    store["demo_simple/files"] = np.asarray(files)
    for fn in files:
        rv, rf = ours.read_obj(os.path.join(ref.results_dir, fn))
        assert np.array_equal(rf, f), fn                                  # the template's faces
        store_sampled(store, "demo_simple/" + fn, rv)


def reference_fit_loop(store, h, tmp):
    import types as T_
    from oracle import tf1_shim as S
    N = TR.FIT_N
    data = TR.fit_data()
    tag, cfg, _, step = G.configs()[0]
    params, batch = G.inputs(cfg, h, N)
    ref_log = []
    with _stubs():
        class Session(object):
            def __init__(self, *a, **k):
                pass

            def run(self, fetches, feed_dict=None):
                if isinstance(fetches, list) and len(fetches) == 2:
                    by_name = {id(model.ph_data_g): "x_g", id(model.ph_data_d): "x_d", id(model.ph_cond_g): "cond_g",
                               id(model.ph_cond2_g): "cond2_g", id(model.ph_cond_d): "cond_d", id(model.ph_cond2_d): "cond2_d"}
                    ref_log.append(("run", {by_name[id(k)]: np.asarray(v) for k, v in feed_dict.items() if id(k) in by_name}))
                    return 1e-3, 0.5
                return None

            def close(self):
                pass

        S.install(template_vertices=np.zeros((6890, 3)))
        S.SESSION_FACTORY = Session
        feeds = dict(data_g=batch["x_g"], data_d=batch["x_d"], condition_g=batch["cond_g"], condition2_g=batch["cond2_g"],
                     condition_d=batch["cond_d"], condition2_d=batch["cond2_d"], gt=batch["gt"], eps=batch["eps"])
        S.reset(feeds=feeds, params=params, global_step=0)
        with contextlib.redirect_stdout(io.StringIO()):
            from lib import models as RM
            kw = G.reference_kwargs(cfg, h, N, name="fitloop")
            kw["num_epochs"] = 2
            model = RM.CAPE(**kw)
            model.build_graph(model.input_num_verts, model.nn_input_channel, phase="train")
            model._get_path = lambda folder: os.path.join(tmp, "ref", folder, "fitloop")
            model.evaluate = lambda *a, **k: (ref_log.append(("validate", None)) or ("", 0.25, 0.0, 0.0))
            model.op_saver = T_.SimpleNamespace(save=lambda sess, path, global_step=None: ref_log.append(("save", global_step)))
            np.random.seed(11)
            ref_losses, _ = model.fit(data)
    # every fed batch is made of rows of the training arrays: stored as those row numbers
    rows = []
    for kind, arg in ref_log:
        if kind == "run":
            r = []
            for k in TR.FIT_FEEDS:
                src = getattr(data, TR.FIT_SOURCE[k])
                r.append([next(i for i in range(len(src)) if np.array_equal(x, src[i])) for x in arg[k]])
                assert np.array_equal(src[r[-1]], arg[k]), k
            rows.append(r)
    store["fit/events"] = np.asarray([e[0] for e in ref_log])
    store["fit/saves"] = np.asarray([e[1] for e in ref_log if e[0] == "save"], np.int64)
    store["fit/rows"] = np.asarray(rows, np.int64)
    store["fit/losses"] = np.asarray(ref_losses, np.float64)


def reference_predict_loop(store, h):
    from oracle import tf1_shim as S
    N = TR.LOOP_N
    data, cond, cond2, labels = TR.predict_data()
    tag, cfg, _, step = G.configs()[0]
    params, batch = G.inputs(cfg, h, N)
    with _stubs():
        class Session(object):
            def __init__(self, *a, **k):
                pass

            def run(self, fetches, feed_dict=None):
                x = np.asarray(feed_dict[model.ph_data_g], np.float32)
                c = np.asarray(feed_dict[model.ph_cond_g], np.float32)
                if isinstance(fetches, list):
                    l = TR.losses_of(x)
                    return TR.out_of(x, c), l[0], l[1], l[2]
                return TR.out_of(x, c)

        S.install(template_vertices=np.zeros((6890, 3)))
        feeds = dict(data_g=batch["x_g"], data_d=batch["x_d"], condition_g=batch["cond_g"], condition2_g=batch["cond2_g"],
                     condition_d=batch["cond_d"], condition2_d=batch["cond2_d"], gt=batch["gt"], eps=batch["eps"])
        S.reset(feeds=feeds, params=params, global_step=0)
        with contextlib.redirect_stdout(io.StringIO()):
            from lib import models as RM
            model = RM.CAPE(**G.reference_kwargs(cfg, h, N, name="predloop"))
            model.build_graph(model.input_num_verts, model.nn_input_channel, phase="train")
            ref_pred, ref_r, ref_l, ref_e = model.predict(data, cond, cond2, labels, sess=Session())
            try:
                model.predict(data, cond, cond2, None, sess=Session())
                raise AssertionError("the reference's predict without labels was expected to raise IndexError")
            except IndexError:
                pass
            ref_string = model.evaluate(data, cond, cond2, labels, sess=Session())
    store_sampled(store, "predict/pred", ref_pred)
    store["predict/losses"] = np.asarray([ref_r, ref_l, ref_e], np.float64)
    store["predict/evaluate_line"] = np.asarray(ref_string[0])
    store["predict/evaluate_values"] = np.asarray(ref_string[1:], np.float64)


def reference_encode_decode_loops(store, h):
    from oracle import tf1_shim as S
    N = TR.LOOP_N
    data, cond, cond2, zt, ye, y2e = TR.encdec_data()
    f_mean, f_var, f_c, f_c2, f_dec = TR.encdec_standins()
    tag, cfg, _, step = G.configs()[0]
    params, batch = G.inputs(cfg, h, N)
    size = len(data)
    with _stubs():
        class Session(object):
            def __init__(self, *a, **k):
                pass

            def run(self, fetches, feed_dict=None):
                fd = {id(k): np.asarray(v, np.float32) for k, v in feed_dict.items() if not isinstance(v, bool)}
                g = lambda ph: fd[id(ph)]
                if not isinstance(fetches, list):
                    return f_dec(g(model.ph_z_total), g(model.ph_y_latent), g(model.ph_y2_latent))
                if len(fetches) == 4:
                    return f_mean(g(model.ph_data_g)), f_var(g(model.ph_data_g)), f_c(g(model.ph_cond_g)), f_c2(g(model.ph_cond2_g))
                return f_c(g(model.ph_cond_g)), f_c2(g(model.ph_cond2_g))

        S.install(template_vertices=np.zeros((6890, 3)))
        S.SESSION_FACTORY = Session
        feeds = dict(data_g=batch["x_g"], data_d=batch["x_d"], condition_g=batch["cond_g"], condition2_g=batch["cond2_g"],
                     condition_d=batch["cond_d"], condition2_d=batch["cond2_d"], gt=batch["gt"], eps=batch["eps"])
        feeds.update(G.demo_feeds(cfg, N))
        S.reset(feeds=feeds, params=params, global_step=0)
        with contextlib.redirect_stdout(io.StringIO()):
            from lib import models as RM
            model = RM.CAPE(**G.reference_kwargs(cfg, h, N, name="encdec"))
            model.build_graph(model.input_num_verts, model.nn_input_channel, phase="demo")
            ref_enc = model.encode(data, cond, cond2)
            ref_cond = model.encode_only_condition(cond, cond2)
            ref_dec = model.decode(zt, cond=np.tile(ye, (size, 1)), cond2=np.tile(y2e, (size, 1)))
            ref_dec1 = model.decode(zt, cond=ye, cond2=y2e)
    for i, a in enumerate(ref_enc):
        store["encode/%d" % i] = a
    for i, a in enumerate(ref_cond):
        store["encode_only_condition/%d" % i] = a
    store["decode/tiled"], store["decode/one_row"] = ref_dec, ref_dec1


def reference_learning_rates(store):
    import types as T_
    from oracle import tf1_shim as S
    lrs, steps_after = [], []
    with _stubs():
        S.install(template_vertices=np.zeros((6890, 3)))
        from lib import models as RM
        for warm in (True, False):
            cfg = TR.lr_config(warm)
            for step in TR.LR_STEPS:
                S.reset(params={"generator/w": np.ones(3, np.float32), "discriminator/w": np.ones(3, np.float32)},
                        global_step=step)
                tf = S.tf
                with tf.variable_scope("generator"):
                    wg = tf.get_variable("w", [3])
                with tf.variable_scope("discriminator"):
                    wd = tf.get_variable("w", [3])
                me = T_.SimpleNamespace(lr_warmup=warm, optim_condnet=True)
                with contextlib.redirect_stdout(io.StringIO()):
                    RM.CAPE.training(me, loss_g=(wg * wg).sum(), loss_d=(wd * wd).sum(), lr_g=cfg["lr"],
                                     lr_d=cfg["lr"] * cfg["lr_scaler"], optimizer="sgd", decay_steps=cfg["decay_steps"],
                                     decay_rate=cfg["decay_rate"], momentum=0.9)
                S.run_pending()
                lrs.append(np.asarray(S.RECORD["lr"], np.float64))
                steps_after.append(int(S.GLOBAL_STEP))
    store["lr/values"] = np.asarray(lrs).reshape(2, len(TR.LR_STEPS), -1)
    store["lr/global_step_after"] = np.asarray(steps_after, np.int64).reshape(2, len(TR.LR_STEPS))


def main():
    if not os.path.isdir(os.path.join(G.REF, "lib")):
        sys.exit("set CAPE_REFERENCE to a checkout of the reference")
    from cape_b200 import topology as T
    L, D, U, p, L_d, D_d, _ = T.load_graph_mtx(load_for_demo=True)
    h = dict(L=L, D=D, U=U, p=p, L_d=L_d, D_d=D_d)
    with open(OUT_JSON, "w") as f:
        json.dump(reference_config(), f, indent=1, sort_keys=True)
        f.write("\n")
    store = {}
    with tempfile.TemporaryDirectory() as tmp:
        reference_body_data(store, tmp)
        reference_demo_simple(store, tmp)
        reference_fit_loop(store, h, tmp)
    reference_predict_loop(store, h)
    reference_encode_decode_loops(store, h)
    reference_learning_rates(store)
    np.savez_compressed(OUT_NPZ, **store)
    for fn in (OUT_JSON, OUT_NPZ):
        print("wrote", fn, os.path.getsize(fn), "bytes")


if __name__ == "__main__":
    main()
