"""ImageNet classifiers (Darknet-19, Darknet-53): [avgpool], [softmax], [cost] in the parser, the port and the engine, and the
batched top-k entry points.  CPU tests need no GPU; the GPU ones are marked and compare outputs only.

Tolerances are those of tests/test_gpu_parity.py: fp32 mode 1e-4 * max|ref| per layer, bf16 teacher-forced 1e-2 * max|ref|,
bf16 free-running within the bf16 storage error model (3e-2 max, 2e-2 rms of max|ref|)."""
import ctypes
import hashlib
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import np_classifier as C
from conftest import model_files

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from oracle import np_darknet as P  # noqa: E402
from oracle import ref_darknet as R  # noqa: E402
from yolo_tensorflow_b200 import synth  # noqa: E402

TABLES = os.path.join(REPO, "tests", "golden", "layer_tables")
CLASSIFIERS = ["darknet19", "darknet53"]
# darknet's FLOP formula (2 * filters * size^2 * channels * out_h * out_w per convolution) over the cfg tables
FLOPS = {"darknet53": 18_570_231_808, "darknet19": 5_581_979_648}
FP32_TOL, BF16_LAYER_TOL, BF16_E2E_TOL, BF16_E2E_RMS_TOL = 1e-4, 1e-2, 3e-2, 2e-2

PARSE = textwrap.dedent("""
    import sys
    sys.path.insert(0, %r)
    from yolo_tensorflow_b200 import darknet as dn
    net = dn.Network(sys.argv[1])
    print(net.n, net.batch, net.w, net.h)
    for L in net.layers:
        print(L["type_name"], L["out_w"], L["out_h"], L["out_c"], L["inputs"], L["outputs"])
    if len(sys.argv) > 2:
        print("resize", net.resize(int(sys.argv[2]), int(sys.argv[2])), net.w, net.h)
        for L in net.layers:
            print(L["type_name"], L["w"], L["h"], L["out_w"], L["out_h"], L["out_c"], L["inputs"], L["outputs"])
    net.close()
""" % REPO)


def run_parse(cfg, *extra):
    return subprocess.run([sys.executable, "-c", PARSE, cfg, *extra], capture_output=True, text=True)


def tail_cfg(tmp_path, tail, name="t.cfg"):
    """a 16x16 two-layer body followed by `tail` sections"""
    p = tmp_path / name
    p.write_text("[net]\nbatch=1\nheight=16\nwidth=16\nchannels=3\n"
                 "[convolutional]\nbatch_normalize=1\nfilters=32\nsize=3\nstride=1\npad=1\nactivation=leaky\n"
                 "[convolutional]\nfilters=40\nsize=1\nstride=1\npad=1\nactivation=linear\n" + tail)
    return str(p)


# ---------------------------------------------------------------------------------------------------
# CPU: parser, cfgs, synthetic weights, port
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", CLASSIFIERS)
def test_classifier_layer_table_matches_golden(model):
    r = run_parse(os.path.join(REPO, "cfg", model + ".cfg"))
    assert r.returncode == 0, r.stderr
    assert r.stderr.splitlines() == open(os.path.join(TABLES, model + ".txt")).read().splitlines()
    rows = r.stdout.splitlines()
    n = int(rows[0].split()[0])
    layers = [x.split() for x in rows[1:]]
    assert n == {"darknet53": 79, "darknet19": 27}[model] == len(layers)
    tail = ["CONVOLUTIONAL", "AVGPOOL"] if model == "darknet19" else ["AVGPOOL", "CONVOLUTIONAL"]
    assert [x[0] for x in layers[-4:]] == tail + ["SOFTMAX", "COST"]
    assert layers[-2][5] == "1000" and layers[-1][5] == "1000"       # softmax outputs; cost passes them on
    assert "avg  " in r.stderr and "softmax" in r.stderr and "cost" in r.stderr


@pytest.mark.parametrize("model", CLASSIFIERS)
def test_classifier_bflops_match_darknets_formula(model):
    r = run_parse(os.path.join(REPO, "cfg", model + ".cfg"))
    printed = sum(float(x.split()[-2]) for x in r.stderr.splitlines() if x.endswith("BFLOPs"))
    assert abs(printed - FLOPS[model] / 1e9) < 0.0005 * r.stderr.count("BFLOPs")      # each row is rounded to 3 decimals
    shapes = synth.walk_shapes(os.path.join(REPO, "cfg", model + ".cfg"))["layers"]
    exact = sum(2 * L["n"] * L["size"] ** 2 * L["c"] * L["out"][1] * L["out"][2] for L in shapes if L["type"] == "convolutional")
    assert exact == FLOPS[model]


def test_classifier_cfgs_are_derived_and_existing_cfgs_unchanged(tmp_path):
    """cfg/derive_cfgs.py writes the committed cfgs byte for byte, the four detection cfgs included"""
    sys.path.insert(0, os.path.join(REPO, "cfg"))
    import derive_cfgs
    for name, fn in derive_cfgs.MODELS.items():
        assert fn() == open(os.path.join(REPO, "cfg", name + ".cfg")).read(), name


@pytest.mark.parametrize("model", CLASSIFIERS)
def test_reference_parser_agrees_on_classifiers_when_available(model):
    """the three format strings (avgpool_layer.c, softmax_layer.c, cost_layer.c) were quoted, not compiled, here: the
    reference parser pins them wherever oracle/_ref is built"""
    if not R.available():
        pytest.skip("oracle/_ref is not built")
    code = ("import ctypes, sys; lib = ctypes.CDLL(%r); lib.parse_network_cfg.restype = ctypes.c_void_p; "
            "lib.parse_network_cfg.argtypes = [ctypes.c_char_p]; lib.parse_network_cfg(sys.argv[1].encode())" % R.REF_SO)
    cfg = os.path.join(REPO, "cfg", model + ".cfg")
    ref = subprocess.run([sys.executable, "-c", code, cfg], capture_output=True, text=True)
    assert ref.stderr == run_parse(cfg).stderr


def test_softmax_groups_and_temperature_are_parsed(tmp_path):
    cfg = tail_cfg(tmp_path, "[avgpool]\n[softmax]\ngroups=4\ntemperature=2.5\n[cost]\ntype=sse\n")
    r = run_parse(cfg)
    assert r.returncode == 0, r.stderr
    assert "softmax                                        %4d\n" % 40 in r.stderr
    assert "Unused field" not in r.stderr
    port = C.Net(cfg)
    assert port.layers[3].groups == 4 and port.layers[3].temperature == 2.5


@pytest.mark.parametrize("tail,message", [
    ("[avgpool]\n[softmax]\ntree=data/9k.tree\n", "softmax tree="),
    ("[avgpool]\n[softmax]\nspatial=1\n", "softmax spatial="),
    ("[avgpool]\n[softmax]\ngroups=3\n", "softmax groups must divide"),
    ("[avgpool]\n[softmax]\n[avgpool]\n", "Layer before avgpool layer must output image."),
])
def test_unsupported_classifier_options_exit_with_a_message(tmp_path, tail, message):
    r = run_parse(tail_cfg(tmp_path, tail))
    assert r.returncode != 0 and message in r.stderr


def test_resize_network_refuses_a_classifier_and_changes_nothing():
    r = run_parse(os.path.join(REPO, "cfg", "darknet53.cfg"), "320")
    rows = r.stdout.splitlines()
    k = next(i for i, x in enumerate(rows) if x.startswith("resize"))
    assert rows[k] == "resize -1 256 256"
    assert "Cannot resize this type of layer" in r.stderr
    before = [x.split() for x in rows[1:k]]
    after = [x.split() for x in rows[k + 1:]]
    assert [a[:1] + a[3:] for a in after] == before


def test_detection_weight_files_are_unchanged(tmp_path):
    """the classifier damping leaves the synthetic files of the detection models as they were"""
    want = {"yolov3-tiny": "163ad846242c7578198ba804547e23e436778a06d1a401a6f9f30511d6902264",
            "yolov2": "50770053d741c7437e3e47be3fba52575159c5db8f847f23991f2b0b0ccfda00"}
    for model, digest in want.items():
        cfg = synth.make_cfg(model, str(tmp_path), batch=2, width=96, height=96)
        w = str(tmp_path / (model + ".weights"))
        synth.write_weights(cfg, w, seed=0, damp_heads=True)
        assert hashlib.sha256(open(w, "rb").read()).hexdigest() == digest, model


def test_classifier_weights_give_unsaturated_probabilities(tmp_path):
    cfg = synth.make_cfg("darknet19", str(tmp_path), batch=2, width=64, height=64)
    w = str(tmp_path / "d19.weights")
    synth.write_weights(cfg, w, seed=0)
    assert len(synth.walk_shapes(cfg)["layers"]) == 27
    outs = C.Net(cfg, w).forward(synth.make_images(2, 3, 64, 64, 1000))
    probs = outs[-1]
    assert np.allclose(probs.sum(axis=1), 1, atol=1e-5)
    assert 1e-3 < probs.max() < .9                                   # neither uniform nor one-hot
    assert np.array_equal(outs[-1], outs[-2])                        # [cost] is an identity


def test_port_softmax_against_float64():
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((3, 24)) * 4).astype(np.float32)
    for groups, temp in ((1, 1.), (4, 1.), (3, 2.5), (2, .7)):
        L = P.Layer(inputs=24, groups=groups, temperature=temp)
        got = C.fwd_softmax(None, L, x, [])
        v = x.reshape(3, groups, -1).astype(np.float64) / temp
        e = np.exp(v - v.max(axis=2, keepdims=True))
        want = (e / e.sum(axis=2, keepdims=True)).reshape(3, -1)
        assert np.abs(got - want).max() <= 1e-6, (groups, temp)


def test_port_avgpool_is_the_mean():
    x = np.random.default_rng(6).standard_normal((2, 5, 7, 3)).astype(np.float32)
    L = P.Layer(c=5, h=7, w=3)
    got = C.fwd_avgpool(None, L, x, [])
    assert got.shape == (2, 5, 1, 1)
    assert np.abs(got[:, :, 0, 0] - x.astype(np.float64).mean(axis=(2, 3))).max() <= 1e-6


def top_k_rows():
    rng = np.random.default_rng(7)
    rows = [rng.random(50).astype(np.float32) for _ in range(6)]
    planted = rng.random(50).astype(np.float32)
    planted[[3, 11, 40]] = planted.max() + 1                         # a three-way tie at the top
    planted[[5, 6]] = planted[20]                                    # and one further down
    zeros = np.zeros(50, np.float32)
    zeros[[7, 30]] = .5
    few = np.round(rng.random(50) * 4).astype(np.float32) / 4        # five distinct values, many ties
    return np.stack(rows + [planted, zeros, np.zeros(50, np.float32), few, -zeros])


def test_port_top_k_is_the_insertion_loop():
    """top_k of utils.c: descending values (those of a stable argsort), and with distinct values the stable argsort's indices.
    Among equal values the loop's own order: an entry displaced from a slot moves on only past strictly smaller ones"""
    for row in top_k_rows():
        for k in (1, 3, 5, 17, 50):
            got = C.top_k(row, k)
            order = np.argsort(-row, kind="stable")[:k]
            assert np.array_equal(row[got], row[order])
            if len(np.unique(row)) == len(row):
                assert np.array_equal(got, order)
            assert len(set(got.tolist())) == k
    assert C.top_k(np.array([5, 5, 3, 6], np.float32), 3).tolist() == [3, 1, 0]
    assert C.top_k(np.array([5, 5, 3, 6], np.float32), 4).tolist() == [3, 1, 0, 2]


def test_library_top_k_equals_the_port():
    from yolo_tensorflow_b200 import darknet as dn
    for row in top_k_rows():
        for k in (1, 5, 20):
            idx = (ctypes.c_int * k)()
            dn.lib.top_k(row.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), len(row), k, idx)
            assert list(idx) == C.top_k(row, k).tolist()


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dn():
    from yolo_tensorflow_b200 import darknet
    return darknet


def open_net(dn, model, batch, size, workdir, prec, fuse=None):
    cfg, wpath = model_files(model, batch, size, workdir)
    fd = os.dup(2); devnull = os.open(os.devnull, os.O_WRONLY); os.dup2(devnull, 2)
    try:
        net = dn.Network(cfg, wpath, precision=prec, fuse=fuse)
    finally:
        os.dup2(fd, 2); os.close(fd); os.close(devnull)
    return net, cfg, wpath


def layer_sources(L, i):
    if L.type == "route":
        return L.src
    if L.type == "shortcut":
        return [i - 1, L.src]
    return [i - 1]


def teacher_forced(dn, net, port, x):
    """every layer recomputed from the port's outputs of its inputs; returns [(layer, kernel, err / max|ref|)]"""
    outs = port.forward(x)
    b = x.shape[0]
    net.predict(x)
    res = [(0, net.kernel(0), np.abs(net.layer_output(0) - outs[0].reshape(b, -1)).max() / np.abs(outs[0]).max())]
    for i, L in enumerate(port.layers[1:], 1):
        for j in layer_sources(L, i):
            net.set_layer_output(j, outs[j].reshape(b, -1))
        net.run_layers(i, i + 1)
        a, r = net.layer_output(i), outs[i].reshape(b, -1)
        assert np.isfinite(a).all(), (i, L.type)
        res.append((i, net.kernel(i), np.abs(a - r).max() / np.abs(r).max()))
    return res, outs


@pytest.mark.gpu
@pytest.mark.parametrize("model", CLASSIFIERS)
def test_fp32_teacher_forced_and_free_running(dn, model, workdir):
    net, cfg, wpath = open_net(dn, model, 2, 64, workdir, dn.PREC_FP32, fuse=False)
    port = C.Net(cfg, wpath)
    x = synth.make_images(2, 3, 64, 64, 77)
    res, outs = teacher_forced(dn, net, port, x)
    for i, k, err in res:
        assert err <= FP32_TOL, (i, k, err)
    kernels = {k for _, k, _ in res}
    assert {"avgpool", "softmax", "alias"} <= kernels
    probs = net.predict(x).reshape(2, -1)
    assert np.abs(probs - outs[-1]).max() <= FP32_TOL * np.abs(outs[-1]).max()
    net.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model,size", [("darknet19", 224), ("darknet53", 256)])
def test_bf16_teacher_forced_and_free_running(dn, model, size, workdir):
    net, cfg, wpath = open_net(dn, model, 8, size, workdir, dn.PREC_BF16, fuse=False)
    port = C.Net(cfg, wpath)
    x = synth.make_images(8, 3, size, size, 78)
    res, outs = teacher_forced(dn, net, port, x)
    for i, k, err in res:
        assert err <= BF16_LAYER_TOL, (i, k, err)
    cls_conv = max(i for i, L in enumerate(port.layers) if L.type == "convolutional")
    assert net.kernel(cls_conv) == "conv_tc"                         # the 1000-filter conv on tcgen05
    assert [net.kernel(i) for i in range(net.n) if port.layers[i].type in ("avgpool", "softmax")] == ["avgpool", "softmax"]
    # free running: the logits (the [softmax] input) within the bf16 storage error model, and the ranking where the port's
    # margin is larger than twice the measured logit error
    probs = net.predict(x).reshape(8, -1)
    sm = next(i for i, L in enumerate(port.layers) if L.type == "softmax")
    a, r = net.layer_output(sm - 1), outs[sm - 1].reshape(8, -1)
    scale = np.abs(r).max()
    assert np.abs(a - r).max() <= BF16_E2E_TOL * scale, np.abs(a - r).max() / scale
    assert np.sqrt(((a - r).astype(np.float64) ** 2).mean()) <= BF16_E2E_RMS_TOL * scale
    checked = 0
    for b in range(8):
        err = np.abs(a[b] - r[b]).max()
        srt = np.sort(r[b])[::-1]
        want, got = C.top_k(outs[-1][b], 5), C.top_k(probs[b], 5)
        if srt[0] - srt[1] > 2 * err:
            assert got[0] == want[0], b
            checked += 1
        if srt[4] - srt[5] > 2 * err:
            assert set(got) == set(want), b
    assert checked >= 1
    net.close()


NOT_MATERIALISED = ("conv_tc+shortcut", "conv_tc(block)", "conv_tc+upsample", "conv_stem+maxpool")


@pytest.mark.gpu
@pytest.mark.parametrize("model,size", [("darknet19", 224), ("darknet53", 256)])
def test_headline_plan_teacher_forced_groups(dn, model, size, workdir):
    """the b64 plan the measurement runs (fusion on), one launch or fused group at a time against the port, as
    test_gpu_parity.test_headline_plan_teacher_forced_groups does for the detectors"""
    batch = 64
    net, cfg, wpath = open_net(dn, model, batch, size, workdir, dn.PREC_BF16)
    port = C.Net(synth.make_cfg(model, workdir, batch=2, width=size, height=size), wpath)
    base = synth.make_images(2, 3, size, size, 1005)
    outs = [o.reshape(2, -1) for o in port.forward(base)]
    reps = batch // 2
    x = np.ascontiguousarray(np.concatenate([base] * reps))
    probe = sorted({0, 1, 2, 3, batch // 2, batch // 2 + 1, batch - 2, batch - 1})
    net.predict(x)
    kernels = [net.kernel(i) for i in range(net.n)]
    cls_conv = max(i for i, L in enumerate(port.layers) if L.type == "convolutional")
    assert kernels[cls_conv] == "conv_tc" and "avgpool" in kernels and "softmax" in kernels
    start, checked = 0, 0
    for j, L in enumerate(port.layers):
        if kernels[j] in NOT_MATERIALISED:
            continue
        if start > 0:
            sources = {s for i in range(start, j + 1) for s in layer_sources(port.layers[i], i) if s < start}
            for src in sorted(sources):
                assert kernels[src] not in NOT_MATERIALISED, (j, src)
                net.set_layer_output(src, np.ascontiguousarray(np.tile(outs[src], (reps, 1))))
            net.run_layers(start, j + 1)
        a = net.layer_output(j)[probe]
        r = outs[j][[q % 2 for q in probe]]
        err = np.abs(a - r).max() / np.abs(r).max()
        assert np.isfinite(a).all() and err <= BF16_LAYER_TOL, (j, L.type, kernels[j], err)
        checked += 1
        start = j + 1
    assert checked >= net.n // 2
    net.close()


@pytest.mark.gpu
def test_device_top_k_equals_the_port(dn):
    rows = top_k_rows()
    rng = np.random.default_rng(8)
    wide = rng.random((9, 1000)).astype(np.float32)
    wide[1] = 0.
    wide[2, ::7] = wide[2].max()
    for arr in (rows, wide):
        for k in (1, 5, 17, 50):
            got = dn.top_k_arrays(arr, k)
            want = np.stack([C.top_k(r, k) for r in arr])
            assert np.array_equal(got, want), k
    big = rng.standard_normal((3, 20000)).astype(np.float32)
    assert np.array_equal(dn.top_k_arrays(big, 64), np.stack([C.top_k(r, 64) for r in big]))


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_classify_batch_is_top_k_of_network_predict(dn, prec, workdir):
    p = dn.PREC_FP32 if prec == "fp32" else dn.PREC_BF16
    net, _, _ = open_net(dn, "darknet53", 4, 64, workdir, p)
    x = synth.make_images(4, 3, 64, 64, 90)
    probs = net.predict(x).reshape(4, -1)
    assert np.allclose(probs.sum(axis=1), 1, atol=1e-4)
    for top in (1, 5, 64):
        cls, pr = net.classify_batch(x, top)
        want = np.stack([C.top_k(r, top) for r in probs])
        assert np.array_equal(cls, want), top
        assert np.array_equal(pr, np.take_along_axis(probs, want, axis=1))
    net.close()


@pytest.mark.gpu
def test_batch_results_equal_batch1_results(dn, workdir):
    x = synth.make_images(4, 3, 64, 64, 91)
    big, _, _ = open_net(dn, "darknet19", 4, 64, workdir, dn.PREC_FP32)
    one, _, _ = open_net(dn, "darknet19", 1, 64, workdir, dn.PREC_FP32)
    cls4, pr4 = big.classify_batch(x, 5)
    p4 = big.predict(x).reshape(4, -1)
    for b in range(4):
        cls1, pr1 = one.classify_batch(x[b:b + 1], 5)
        assert np.array_equal(cls1[0], cls4[b]) and np.array_equal(pr1[0], pr4[b])          # fp32: bit for bit
        assert np.array_equal(one.predict(x[b:b + 1]), p4[b])
    big.close(); one.close()
    # bf16 at b64: the same plan at a lower logical batch is bit-identical; two runs are bit-identical
    net, _, _ = open_net(dn, "darknet53", 64, 256, workdir, dn.PREC_BF16)
    x = synth.make_images(64, 3, 256, 256, 92)
    c1, p1 = net.classify_batch(x, 5)
    c2, p2 = net.classify_batch(x, 5)
    assert np.array_equal(c1, c2) and p1.tobytes() == p2.tobytes()
    dn.set_batch_network(net.ptr, 1)
    net.batch = 1
    c0, q0 = net.classify_batch(x[5:6], 5)
    assert np.array_equal(c0[0], c1[5]) and np.array_equal(q0[0], p1[5])
    net.close()


@pytest.mark.gpu
def test_serving_loops_equal_the_synchronous_call(dn, workdir):
    net, _, _ = open_net(dn, "darknet19", 4, 224, workdir, dn.PREC_BF16)
    batches = [np.ascontiguousarray(synth.make_images(4, 3, 224, 224, 200 + k)) for k in range(3)]
    want = [net.classify_batch(b, 5) for b in batches]
    cls = np.zeros((4, 5), np.int32); pr = np.zeros((4, 5), np.float32)
    cp, pp = cls.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), pr.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    dn.lib.b200_submit_batch(net.ptr, batches[0].ctypes.data_as(ctypes.c_void_p))
    for k in range(3):
        nxt = batches[k + 1].ctypes.data_as(ctypes.c_void_p) if k < 2 else None
        assert dn.lib.b200_classify_submitted(net.ptr, nxt, 5, cp, pp) == 4
        assert np.array_equal(cls, want[k][0]) and np.array_equal(pr, want[k][1]), k
    # resident input: letterbox batch k+1 on the device while batch k is classified
    rng = np.random.default_rng(3)
    pics = [[(rng.random((480, 640, 3)) * 255).astype(np.uint8) for _ in range(4)] for _ in range(3)]
    want = []
    for imgs in pics:
        assert net.letterbox_batch_u8(imgs) == 0
        want.append(net.classify_batch(None, 5))
    RES = ctypes.c_void_p(1)
    net.letterbox_batch_u8(pics[0])
    dn.lib.b200_submit_batch(net.ptr, RES)
    for k in range(3):
        if k < 2:
            net.letterbox_batch_u8(pics[k + 1])
        assert dn.lib.b200_classify_submitted(net.ptr, RES if k < 2 else None, 5, cp, pp) == 4
        assert np.array_equal(cls, want[k][0]) and np.array_equal(pr, want[k][1]), k
    net.close()


@pytest.mark.gpu
def test_python_wrapper_classify_on_ppm(dn, workdir, tmp_path):
    """python/darknet.py classify(): network_predict_image's output, every class, most probable first"""
    net, _, _ = open_net(dn, "darknet19", 1, 224, workdir, dn.PREC_BF16)
    img = (np.random.default_rng(4).random((150, 200, 3)) * 255).astype(np.uint8)
    ppm = tmp_path / "x.ppm"
    with open(ppm, "wb") as f:
        f.write(b"P6\n200 150\n255\n" + img.tobytes())
    names = tmp_path / "n.names"; names.write_text("\n".join(f"c{i}" for i in range(1000)) + "\n")
    data = tmp_path / "c.data"; data.write_text(f"classes=1000\nnames={names}\n")
    meta = dn.load_meta(str(data).encode())
    im = dn.load_image(str(ppm).encode(), 0, 0)
    res = dn.classify(net.ptr, meta, im)
    probs = np.ctypeslib.as_array(dn.predict_image(net.ptr, im), shape=(1000,)).copy()
    assert len(res) == 1000
    assert [v for _, v in res] == sorted(probs.tolist(), reverse=True)
    assert {n for n, _ in res} == {f"c{i}".encode() for i in range(1000)}
    assert all(probs[int(n[1:])] == v for n, v in res)
    dn.free_image(im)
    net.close()


@pytest.mark.gpu
def test_flows_are_bit_identical_to_one_launch_per_layer(dn, workdir):
    os.environ["B200_FLOW"] = "1"
    try:
        net, _, _ = open_net(dn, "darknet53", 16, 256, workdir, dn.PREC_BF16)
    finally:
        os.environ.pop("B200_FLOW", None)
    assert net.flows()
    x = synth.make_images(16, 3, 256, 256, 93)
    net.set_flow(0)
    p0 = net.predict(x); c0 = net.classify_batch(x, 5)
    net.set_flow(1)
    p1 = net.predict(x); c1 = net.classify_batch(x, 5)
    assert p0.tobytes() == p1.tobytes() and np.array_equal(c0[0], c1[0]) and c0[1].tobytes() == c1[1].tobytes()
    net.close()


@pytest.mark.gpu
def test_split_k_plan_matches_the_unsplit_plan(dn, workdir):
    net, _, _ = open_net(dn, "darknet53", 1, 256, workdir, dn.PREC_BF16)
    os.environ["B200_NO_SPLITK"] = "1"
    try:
        ref, _, _ = open_net(dn, "darknet53", 1, 256, workdir, dn.PREC_BF16)
    finally:
        os.environ.pop("B200_NO_SPLITK", None)
    assert any("splitK" in dn.lib.b200_layer_plan(net.ptr, i).decode() for i in range(net.n))
    x = synth.make_images(1, 3, 256, 256, 94)
    sm = next(i for i in range(net.n) if net.layers[i]["type_name"] == "SOFTMAX")
    net.predict(x); ref.predict(x)
    a, r = net.layer_output(sm - 1), ref.layer_output(sm - 1)
    assert np.abs(a - r).max() <= 4e-2 * np.abs(r).max()                # two free-running bf16 pipelines
    assert np.abs(net.layer_output(sm) - ref.layer_output(sm)).max() <= 4e-2 * np.abs(ref.layer_output(sm)).max()
    net.close(); ref.close()


@pytest.mark.gpu
def test_wrong_entry_points_return_minus_one(dn, workdir):
    cls_net, _, _ = open_net(dn, "darknet19", 2, 64, workdir, dn.PREC_BF16)
    x = synth.make_images(2, 3, 64, 64, 95)
    out = (dn.B200_DET * 16)()
    counts = (ctypes.c_int * 2)()
    assert dn.lib.b200_detect_batch(cls_net.ptr, x.ctypes.data_as(ctypes.c_void_p), 64, 64, .5, .45, 1, out, 16, counts) == -1
    assert dn.lib.b200_detect_submitted(cls_net.ptr, None, 64, 64, .5, .45, 1, out, 16, counts) == -1
    cls = np.zeros((2, 64), np.int32); pr = np.zeros((2, 64), np.float32)
    cp, pp = cls.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), pr.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    xp = x.ctypes.data_as(ctypes.c_void_p)
    for top in (0, 65):
        assert dn.lib.b200_classify_batch(cls_net.ptr, xp, top, cp, pp) == -1
    assert dn.lib.b200_classify_batch(cls_net.ptr, xp, 5, cp, pp) == 2                  # still usable
    cls_net.close()
    det, _, _ = open_net(dn, "yolov3", 2, 160, workdir, dn.PREC_BF16)
    assert dn.lib.b200_classify_batch(det.ptr, xp, 5, cp, pp) == -1
    assert dn.lib.b200_classify_submitted(det.ptr, None, 5, cp, pp) == -1
    xd = synth.make_images(2, 3, 160, 160, 95)                         # and the detector still detects
    assert dn.lib.b200_detect_batch(det.ptr, xd.ctypes.data_as(ctypes.c_void_p), 160, 160, .5, .45, 1, out, 16, counts) >= 0
    det.close()
