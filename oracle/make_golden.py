"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN LAYER FILES (TEST INFRASTRUCTURE).

Needs a checkout of tangxyw/RecAlgorithm (the reference):

    python oracle/make_golden.py REFERENCE_CHECKOUT [OUT_DIR]       # OUT_DIR defaults to tests/golden

The five interaction-layer files are imported verbatim from REFERENCE_CHECKOUT/algorithm with
``oracle/tf1_shim`` standing in for TensorFlow 1.14 (see that package's docstring for what
this does and does not pin).  Each fixture stores the seeded inputs, the injected weights
(under the TF variable names the reference created), and the reference outputs computed in
float32 (like the reference) and float64 (anchor).  FM2 and the lookup have no importable
reference function (inline code / TF-internal); their fixtures come from
``oracle/layers_np.py`` and are marked ``source='restated'``.

Beside the fixtures it writes ``reference_digests.json``: the SHA-256 of every array of the run.  The tests need no
reference checkout: they compare the committed fixtures with that record, array by array, and regenerate the restated
fixtures (``gen_restated``, which runs no reference code) bit for bit.
"""
from __future__ import annotations

import hashlib
import importlib.util
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = None                      # REFERENCE_CHECKOUT/algorithm, set by load_reference()
OUT = os.path.join(ROOT, "tests", "golden")
DIGESTS = "reference_digests.json"

sys.path.insert(0, os.path.join(HERE, "tf1_shim"))
sys.path.insert(0, ROOT)
import tensorflow as tf  # noqa: E402  (the shim)

assert "tf1_shim" in tf.__file__, "the TF shim must shadow any real tensorflow"


def _load(relpath, name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, relpath))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_reference(checkout):
    """Import the reference's five interaction-layer files from `checkout` (a tangxyw/RecAlgorithm tree)."""
    global REF, ref_cross, ref_cin, ref_din, ref_senet, ref_bilinear
    REF = os.path.join(os.path.abspath(checkout), "algorithm")
    ref_cross = _load("DCN/cross_layer.py", "ref_cross_layer")
    ref_cin = _load("xDeepFM/cin_layer.py", "ref_cin_layer")
    ref_din = _load("DIN/din_attention.py", "ref_din_attention")
    ref_senet = _load("FiBiNET/senet.py", "ref_senet")
    ref_bilinear = _load("FiBiNET/bilinear_interaction_layer.py", "ref_bilinear")


def fixture_digests(directory):
    """{fixture file: {array name: sha256 of dtype, shape and bytes}} of every .npz in `directory`."""
    out = {}
    for f in sorted(os.listdir(directory)):
        if f.endswith(".npz"):
            with np.load(os.path.join(directory, f), allow_pickle=False) as z:
                out[f] = {k: hashlib.sha256(f"{z[k].dtype.str}{z[k].shape}".encode() + z[k].tobytes()).hexdigest()
                          for k in sorted(z.files)}
    return out


def trunc_normal(rng, shape, std):
    x = rng.standard_normal(shape)
    bad = np.abs(x) > 2
    while bad.any():
        x[bad] = rng.standard_normal(int(bad.sum()))
        bad = np.abs(x) > 2
    return (x * std).astype(np.float32)


def glorot(rng, shape, fan_in=None, fan_out=None):
    fan_in = fan_in or shape[-2]
    fan_out = fan_out or shape[-1]
    lim = (6.0 / (fan_in + fan_out)) ** 0.5
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def run_both(fn, variables):
    """Run ``fn`` (which builds the reference layer) in float32 and float64."""
    outs = {}
    for tag, dt in (("f32", np.float32), ("f64", np.float64)):
        tf.reset(dtype=dt, variables=variables)
        outs[tag] = fn(dt)
    created = tf.created_variables()
    return outs, created


def save(name, **arrays):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez(path, **arrays)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def gen_cross():
    rng = np.random.default_rng(1234)
    for d, L, B in ((82, 1, 8), (82, 3, 8), (480, 3, 6)):
        x0 = trunc_normal(rng, (B, d), 0.25)
        variables = {}
        for i in range(L):
            variables[f"cross_part/wl_{i}"] = glorot(rng, (d, 1))
            variables[f"cross_part/bl_{i}"] = glorot(rng, (d, 1))    # glorot, NOT zeros (cross_layer.py:18-19)

        def fn(dt):
            x0_t = tf.Tensor(x0.astype(dt))
            with tf.variable_scope("cross_part"):              # DCN/dcn.py:156-160
                vec = x0_t
                for i in range(L):
                    vec = ref_cross.cross_layer(x0=x0_t, xl=vec, index=i)
            return vec.a

        outs, created = run_both(fn, variables)
        assert all(created[k] == (d, 1) for k in created)
        ws = np.stack([variables[f"cross_part/wl_{i}"][:, 0] for i in range(L)])
        bs = np.stack([variables[f"cross_part/bl_{i}"][:, 0] for i in range(L)])
        save(f"cross_d{d}_L{L}", x0=x0, ws=ws, bs=bs, out_f32=outs["f32"], out_f64=outs["f64"],
             source="reference:DCN/cross_layer.py via tf1_shim")


def gen_cin():
    rng = np.random.default_rng(2345)
    for m, D, maps, B in ((8, 8, ("50", "50", "50"), 4), (30, 16, ("128", "128"), 3), (8, 16, ("17",), 5)):
        x0 = trunc_normal(rng, (B, m, D), 1.0 / np.sqrt(D))
        variables, hk = {}, m
        for i, h in enumerate(maps):
            h = int(h)
            variables[f"cin_part/cin_layer_{i + 1}_filter"] = glorot(rng, (1, hk * m, h), fan_in=hk * m, fan_out=h)
            hk = h

        def fn(dt):
            x0_t = tf.Tensor(x0.astype(dt))
            outs = []
            with tf.variable_scope("cin_part"):                # xDeepFM/xdeepfm.py:166-174
                xk = x0_t
                for i, h in enumerate(maps):
                    # layer widths reach model_fn as *strings* (xdeepfm.py:253); the reference's
                    # tf.get_variable accepts that because TF int()s shape entries.
                    xk = ref_cin.cin_layer(x0_t, xk, int(h), i + 1)
                    outs.append(xk)
                p_plus = tf.concat([tf.reduce_sum(x, axis=-1) for x in outs], axis=-1)
            return [o.a for o in outs] + [p_plus.a]

        outs, created = run_both(fn, variables)
        arrays = dict(x0=x0, n_layers=len(maps), source="reference:xDeepFM/cin_layer.py via tf1_shim")
        for i in range(len(maps)):
            arrays[f"filter_{i + 1}"] = variables[f"cin_part/cin_layer_{i + 1}_filter"][0]
            arrays[f"x{i + 1}_f32"] = outs["f32"][i]
            arrays[f"x{i + 1}_f64"] = outs["f64"][i]
        arrays["p_plus_f32"] = outs["f32"][-1]
        arrays["p_plus_f64"] = outs["f64"][-1]
        save(f"cin_m{m}_D{D}_" + "x".join(maps), **arrays)


def gen_din():
    rng = np.random.default_rng(3456)
    cases = (("T3_smoke", 2, 3, 4, np.array([0, 1])),          # the reference's own __main__ case (din_attention.py:46-54)
             ("T1", 3, 1, 16, np.array([0, 1, 1])),
             ("T50", 6, 50, 16, np.array([0, 1, 17, 49, 50, 50])))
    for tag, B, T, H, lens in cases:
        q = trunc_normal(rng, (B, H), 0.25)
        keys = trunc_normal(rng, (B, T, H), 0.25)
        variables = {
            "attention_part/f1_att/kernel": glorot(rng, (4 * H, 64)),
            "attention_part/f1_att/bias": (rng.standard_normal(64) * 0.1).astype(np.float32),
            "attention_part/f2_att/kernel": glorot(rng, (64, 32)),
            "attention_part/f2_att/bias": (rng.standard_normal(32) * 0.1).astype(np.float32),
            "attention_part/f3_att/kernel": glorot(rng, (32, 1)),
            "attention_part/f3_att/bias": (rng.standard_normal(1) * 0.1).astype(np.float32),
        }
        arrays = dict(query=q, keys=keys, keys_length=lens.astype(np.int64),
                      source="reference:DIN/din_attention.py via tf1_shim")
        for k, v in variables.items():
            arrays[k.split("/", 1)[1].replace("/", "_")] = v
        for soft in (False, True):
            def fn(dt):
                with tf.variable_scope("attention_part"):      # DIN/din.py:216-218
                    return ref_din.din_attention(tf.Tensor(q.astype(dt)), tf.Tensor(keys.astype(dt)),
                                                 tf.Tensor(lens), is_softmax=soft).a
            outs, _ = run_both(fn, variables)
            arrays[f"out_softmax{int(soft)}_f32"] = outs["f32"]
            arrays[f"out_softmax{int(soft)}_f64"] = outs["f64"]
        save(f"din_{tag}", **arrays)


def gen_fibinet():
    rng = np.random.default_rng(4567)
    for F, K, ratio, B in ((8, 8, 2, 5), (30, 16, 2, 3)):
        x = trunc_normal(rng, (B, F, K), 1.0 / np.sqrt(K))
        r = K // ratio
        variables = {"senet_part/senet_w1": glorot(rng, (F, r)), "senet_part/senet_w2": glorot(rng, (r, F))}

        def fn(dt):
            with tf.variable_scope("senet_part"):              # FiBiNET/fibinet.py:171-174
                return ref_senet.senet(tf.Tensor(x.astype(dt)), embedding_dim=K, reduction_ratio=ratio).a
        outs, created = run_both(fn, variables)
        assert created["senet_part/senet_w1"] == (F, r)        # reduced from K, not F (senet.py:18)
        arrays = dict(x=x, senet_w1=variables["senet_part/senet_w1"], senet_w2=variables["senet_part/senet_w2"],
                      senet_f32=outs["f32"], senet_f64=outs["f64"],
                      source="reference:FiBiNET/{senet,bilinear_interaction_layer}.py via tf1_shim")
        P = (F - 1) * (F - 2) // 2
        for typ, wshape in (("all", (K, K)), ("each", (F - 1, K, K)), ("interaction", (F * (F - 1) // 2, K, K))):
            w = glorot(rng, wshape)
            vs = {f"bilinear_interaction_part/orginal_w_{typ}": w}

            def fn2(dt):
                with tf.variable_scope("bilinear_interaction_part"):   # FiBiNET/fibinet.py:177-181
                    return ref_bilinear.bilinear_interaction_layer(tf.Tensor(x.astype(dt)), embedding_dim=K,
                                                                   type=typ, name="orginal").a
            outs2, created2 = run_both(fn2, vs)
            assert outs2["f32"].shape == (B, P, K), outs2["f32"].shape   # (F-1)(F-2)/2 pairs, not F(F-1)/2
            arrays[f"w_{typ}"] = w
            arrays[f"bilinear_{typ}_f32"] = outs2["f32"]
            arrays[f"bilinear_{typ}_f64"] = outs2["f64"]
        save(f"fibinet_F{F}_K{K}", **arrays)
    # error behaviour: bad type -> ValueError (bilinear_interaction_layer.py:36-38)
    tf.reset()
    try:
        ref_bilinear.bilinear_interaction_layer(tf.Tensor(np.zeros((1, 4, 2), np.float32)), 2, "nope", "x")
        raise AssertionError("reference accepted a bad bilinear type")
    except ValueError:
        pass


def gen_restated():
    from oracle import layers_np as O
    rng = np.random.default_rng(5678)
    for F, D, B in ((6, 8, 16), (40, 32, 8)):
        e = trunc_normal(rng, (B, F, D), 1.0 / np.sqrt(D))
        save(f"fm2_F{F}_D{D}", e=e, out_f32=O.fm2_fwd(e), out_f64=O.fm2_fwd(e.astype(np.float64)),
             pairwise_f64=O.fm2_pairwise(e), source="restated:DeepFM/deepfm.py:184-200")
    # lookup edge cases: OOV, empty string, duplicate ids, empty bag, multi-valued mean
    vocab = [b"userid_8", b"userid_3", b"userid_11", b"userid_5"]
    keys = [b"userid_3", b"", b"userid_999", b"userid_8", b"userid_3", b"userid_5"]
    ids = O.vocab_ids(keys, vocab)
    assert ids.tolist() == [1, -1, -1, 0, 1, 3]
    rows = [4, 3, 5]
    off = np.array([0, 4, 7], dtype=np.int64)
    table = trunc_normal(rng, (sum(rows), 8), 1 / np.sqrt(8))
    ids2 = np.array([[1, 0, 4], [-1, 2, -1], [3, -1, 0], [1, 2, 4], [0, 0, 0], [-1, -1, -1]], dtype=np.int64)
    out = O.embedding_lookup(table, ids2, off)
    bag_ids = np.array([2, 0, -1, 5, 5, -1, -1, 11, 3], dtype=np.int64)
    bag_off = np.array([0, 3, 3, 5, 7, 9], dtype=np.int64)      # bags: [2,0,-1] [] [5,5] [-1,-1] [11,3]
    bag = O.bag_lookup_mean(table, bag_ids, bag_off)
    save("lookup_edge", vocab=np.array(vocab), keys=np.array(keys), key_ids=ids, table=table, field_row_offset=off,
         ids=ids2, out=out, bag_ids=bag_ids, bag_offsets=bag_off, bag_out=bag,
         source="restated:TF1.14 feature_column semantics (SURVEY A.4-A.6) -- parity unpinned")


# ---- inline blocks of model_fns: the cited source lines are read from the reference checkout at generation time and exec()'d ----

class _FakeFC:
    """Stand-in for `tf.feature_column` inside the inline blocks: `fc.input_layer(features, [col])` returns the (B, K)
    embedding injected for that column (the lookup itself is TF-internal and pinned elsewhere as 'unpinned')."""
    @staticmethod
    def input_layer(features, columns):
        return tf.concat([tf.Tensor(features[c]) for c in columns], axis=1)


def exec_ref_lines(relpath, first, last, must_contain, ns):
    import textwrap
    with open(os.path.join(REF, relpath), encoding="utf-8") as fh:
        lines = fh.read().split("\n")[first - 1:last]
    assert must_contain[0] in lines[0] and must_contain[1] in lines[-1], (relpath, lines[0], lines[-1])
    exec(compile(textwrap.dedent("\n".join(lines)), f"{relpath}:{first}-{last}", "exec"), ns)
    return ns


def _inline_case(relpath, first, last, must, e, key, out_name, variables=None, extra=None):
    F = e.shape[1]
    cols = [f"c{f:02d}" for f in range(F)]
    outs = {}
    for tag, dt in (("f32", np.float32), ("f64", np.float64)):
        tf.reset(dtype=dt, variables=variables or {})
        ns = {"tf": tf, "fc": _FakeFC, "features": {c: e[:, f, :].astype(dt) for f, c in enumerate(cols)},
              "params": {key: cols, **(extra or {})}}
        sys.path.insert(0, REF)                              # FwFM imports index_from_upper_triangular from utils.py
        if "index_from_upper_triangular" in must[2:]:
            ns["index_from_upper_triangular"] = _load("utils.py", "ref_utils").index_from_upper_triangular
        exec_ref_lines(relpath, first, last, must, ns)
        outs[tag] = np.asarray(ns[out_name].a if hasattr(ns[out_name], "a") else ns[out_name])
    return outs, tf.created_variables()


def gen_inline():
    from oracle import layers_np as O
    rng = np.random.default_rng(2468)
    for F, D, B in ((6, 8, 16), (40, 32, 8)):
        e = trunc_normal(rng, (B, F, D), 1.0 / np.sqrt(D))
        outs, _ = _inline_case("DeepFM/deepfm.py", 184, 200, ("fields_embeddings = []", "keepdims=True)"), e,
                               "second_order_feature_columns", "fm_second_order_logit")
        save(f"fm2_ref_F{F}_D{D}", e=e, out_f32=outs["f32"], out_f64=outs["f64"], source="reference-executed:DeepFM/deepfm.py:184-200")
        outs, _ = _inline_case("NFM/nfm.py", 155, 168, ('variable_scope("bi_interaction_part")', "nfm = 0.5 *"), e,
                               "category_feature_columns", "nfm")
        save(f"nfm_bi_F{F}_D{D}", e=e, out_f32=outs["f32"], out_f64=outs["f64"], source="reference-executed:NFM/nfm.py:155-168")
    for F, D, B in ((6, 8, 16), (30, 16, 8)):
        e = trunc_normal(rng, (B, F, D), 1.0 / np.sqrt(D))
        P = F * (F - 1) // 2
        r = glorot(rng, (P,), fan_in=P, fan_out=P)
        outs, created = _inline_case("FwFM/fwfm.py", 140, 158, ("fields_embeddings = []", ")", "index_from_upper_triangular"), e,
                                     "second_order_feature_columns", "fwfm_second_order_logit",
                                     variables={"fields_pair_strength/fields_pair_strength_weight": r})
        assert created == {"fields_pair_strength/fields_pair_strength_weight": (P,)}, created
        save(f"fwfm_F{F}_D{D}", e=e, r=r, out_f32=outs["f32"], out_f64=outs["f64"], source="reference-executed:FwFM/fwfm.py:140-158")
    for F, D, t, B in ((5, 8, 4, 16), (30, 16, 8, 6)):
        e = trunc_normal(rng, (B, F, D), 1.0)
        w, b, h, pv = glorot(rng, (D, t)), glorot(rng, (t,), fan_in=t, fan_out=t), glorot(rng, (t, 1)), glorot(rng, (D, 1))
        variables = {"attention_part/attention_w": w, "attention_part/attention_b": b, "attention_part/attention_h": h,
                     "prediction_score_part/p": pv}
        res = {}
        for name in ("weighted_sum", "afm_logit", "attention_score"):
            outs, created = _inline_case("AFM/afm.py", 152, 188, ('variable_scope("pair_interaction_part")', "afm_logit = tf.matmul"), e,
                                         "category_feature_columns", name, variables=variables,
                                         extra={"embedding_dim": D, "attention_factor": t})
            res[name] = outs
        assert created == {"attention_part/attention_w": (D, t), "attention_part/attention_b": (t,),
                           "attention_part/attention_h": (t, 1), "prediction_score_part/p": (D, 1)}, created
        save(f"afm_F{F}_D{D}_t{t}", e=e, w=w, b=b, h=h, p=pv, pooled_f32=res["weighted_sum"]["f32"], pooled_f64=res["weighted_sum"]["f64"],
             logit_f32=res["afm_logit"]["f32"], logit_f64=res["afm_logit"]["f64"], score_f64=res["attention_score"]["f64"],
             source="reference-executed:AFM/afm.py:152-188")


def gen_bst():
    """BST/transformer_layer.py imported verbatim (it does `from leakyrelu import leakyrelu`: BST/ goes on sys.path)."""
    from oracle import layers_np as O
    sys.path.insert(0, os.path.join(REF, "BST"))
    ref_bst = _load("BST/transformer_layer.py", "ref_bst_transformer")
    rng = np.random.default_rng(1357)
    for name, (B, T, d, H, maxlen, lengths) in {"bst_T3_smoke": (2, 3, 4, 3, 5, [0, 1]),               # the file's own __main__ shapes
                                                 "bst_T51_d8_h3": (6, 51, 8, 3, 51, [51, 1, 17, 0, 50, 33]),
                                                 "bst_T20_d16_h2": (4, 20, 16, 2, 24, [20, 7, 0, 13])}.items():
        x = trunc_normal(rng, (B, T, d), 1.0)
        shapes = O.bst_param_shapes(d, H, maxlen)
        p = {"position_embedding": trunc_normal(rng, shapes["position_embedding"], 0.3),
             "w_q": glorot(rng, shapes["w_q"]), "w_k": glorot(rng, shapes["w_k"]), "w_v": glorot(rng, shapes["w_v"]),
             "w_o": glorot(rng, shapes["w_o"]), "ln1_beta": trunc_normal(rng, (d,), 0.1), "ln1_gamma": 1 + trunc_normal(rng, (d,), 0.1),
             "dense_kernel": glorot(rng, (d, d)), "dense_bias": trunc_normal(rng, (d,), 0.1),
             "ln2_beta": trunc_normal(rng, (d,), 0.1), "ln2_gamma": 1 + trunc_normal(rng, (d,), 0.1)}
        variables = {"position_embedding": p["position_embedding"], "w_q_0": p["w_q"], "w_k_0": p["w_k"], "w_v_0": p["w_v"],
                     "w_o_0": p["w_o"], "LayerNorm/beta": p["ln1_beta"], "LayerNorm/gamma": p["ln1_gamma"],
                     "dense/kernel": p["dense_kernel"], "dense/bias": p["dense_bias"],
                     "LayerNorm_1/beta": p["ln2_beta"], "LayerNorm_1/gamma": p["ln2_gamma"]}
        klen = np.asarray(lengths, dtype=np.int64)

        def fn(dt):
            t = tf.Tensor(x.astype(dt))
            return ref_bst.bst_transformer(queries=t, keys=t, values=t, keys_length=tf.Tensor(klen), heads=H, index=0,
                                           max_length=maxlen, use_position_embedding=True).a
        outs, created = run_both(fn, variables)
        assert created == {k: tuple(np.shape(v)) for k, v in variables.items()}, created
        save(name, x=x, keys_length=klen, heads=np.int64(H), max_length=np.int64(maxlen), out_f32=outs["f32"], out_f64=outs["f64"],
             **{f"p_{k}": v for k, v in p.items()}, source="reference-executed:BST/transformer_layer.py:6-79")


def gen_ffm():
    """FFM/ffm.py:145-160 executed with per-field (F-1, |V_i|, K) variables and the id vectors standing in for the one-hot ->
    sparse conversion of :141-144 (to_sparse_tensor + safe_embedding_lookup_sparse == row lookup, empty row -> zeros)."""
    rng = np.random.default_rng(8642)
    for F, K, B in ((4, 4, 9), (5, 8, 16), (9, 16, 6)):
        sizes = [int(v) for v in rng.integers(3, 9, size=F)]
        emb = [trunc_normal(rng, (F - 1, sizes[f], K), 0.5) for f in range(F)]
        ids = np.stack([rng.integers(-1, sizes[f], size=B) for f in range(F)], axis=1).astype(np.int64)
        outs = {}
        for tag, dt in (("f32", np.float32), ("f64", np.float64)):
            tf.reset(dtype=dt)
            ns = {"tf": tf, "params": {"one_hot_category_feature_columns": list(range(F))},
                  "embedding_variables": [tf.Tensor(e.astype(dt)) for e in emb], "field_sparse_ids_list": [ids[:, f] for f in range(F)]}
            exec_ref_lines("FFM/ffm.py", 145, 160, ("second_order_vec = 0.0", "second_order_vec += tf.reduce_sum"), ns)
            outs[tag] = np.asarray(ns["second_order_vec"].a)
        tile = np.zeros((B, F, F - 1, K), np.float32)                         # the (field, slot) layout our lookup produces
        for f in range(F):
            ok = ids[:, f] >= 0
            tile[ok, f] = emb[f][:, ids[ok, f], :].transpose(1, 0, 2)
        save(f"ffm_F{F}_K{K}", ids=ids, tile=tile, out_f32=outs["f32"], out_f64=outs["f64"],
             **{f"emb_{f}": emb[f] for f in range(F)}, source="reference-executed:FFM/ffm.py:145-160")


if __name__ == "__main__":
    if len(sys.argv) not in (2, 3):
        raise SystemExit(__doc__)
    load_reference(sys.argv[1])
    if len(sys.argv) == 3:
        OUT = sys.argv[2]
    gen_cross()
    gen_cin()
    gen_din()
    gen_fibinet()
    gen_restated()
    gen_inline()
    gen_bst()
    gen_ffm()
    with open(os.path.join(OUT, DIGESTS), "w") as fh:
        json.dump(fixture_digests(OUT), fh, indent=1, sort_keys=True)
        fh.write("\n")
