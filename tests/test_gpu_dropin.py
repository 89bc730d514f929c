"""Drop-in claims of INTEGRATION.md, executed: the objects riser.py builds from FILES, the reference's own
(unmodified) control loop driving riser_b200's Model + SignalProcessor, and the input dtypes
SignalProcessor.mad_normalise accepts.  Needs a B200."""
import logging
import os

import numpy as np
import pytest
import torch
import yaml

from riser_b200 import Kit, SignalProcessor, Model, sim, synth
from riser_b200.config import get_config, CNN_SHIPPED
from oracle import refshim
from oracle import control_oracle as ctl
from oracle import preprocess_oracle as pp
from oracle import convnet_oracle as net
from tests.golden import make_golden_params as P

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")


def _write_model_files(tmp_path, target, kit="RNA002", pore="R9.4.1"):
    """model/{target}_model_{kit}_{pore}.pth + model/{target}_config_{kit}_{pore}.yaml as riser.py:39-40 names them;
    the YAML has the layout of riser/model/*_config_*.yaml (model / training keys / cnn block)."""
    d = tmp_path / "model"
    d.mkdir(exist_ok=True)
    pth = synth.save_state_dict(synth.TARGET_SEEDS[target], str(d / f"{target}_model_{kit}_{pore}.pth"))
    cfg = {"model": "cnn", "n_epochs": 30, "batch_size": 32, "learning_rate": 0.0001, "cnn": dict(CNN_SHIPPED)}
    yml = str(d / f"{target}_config_{kit}_{pore}.yaml")
    with open(yml, "w") as f:
        yaml.safe_dump(cfg, f)
    return pth, yml


def test_model_from_pth_path_and_yaml_path(tmp_path):
    """riser.py:35-42 get_models: Model(model_file, get_config(config_file), logger, target)."""
    pth, yml = _write_model_files(tmp_path, "mRNA")
    model = Model(pth, get_config(yml), LOG, "mRNA")
    assert model.target == "mRNA" and model.device.type == "cuda"
    proc = SignalProcessor(Kit.create_from_version("RNA002"))
    x = synth.body_batch(11, 2, 9000)[1]
    sig = proc.mad_normalise(x)
    p_off, p_on = model.classify(sig)                      # control.py:69
    want = net.classify(synth.state_dict(0), pp.mad_normalise(x)).numpy()
    assert abs(p_on.item() - want[1]) < 1e-3 and abs(p_off.item() - want[0]) < 1e-3
    # same weights through the dict route: bit-identical probabilities
    again = Model(synth.state_dict(0), get_config(yml), LOG, "mRNA").classify(sig)
    assert torch.equal(again.cpu(), torch.stack([p_off, p_on]).cpu())
    with pytest.raises(FileNotFoundError):
        Model(str(tmp_path / "missing.pth"), get_config(yml), LOG, "mRNA")


@pytest.mark.parametrize("mode", ["deplete", "enrich"])
def test_reference_control_loop_drives_riser_b200_objects(golden_dir, tmp_path, mode):
    """INTEGRATION.md, import swap: the reference's serial SequencerControl.target (riser/control.py:11-124, restated
    call for call in oracle/control_oracle.serial_target) with riser_b200.Model / SignalProcessor behind it reproduces
    the rows, unblock and stop-receiving calls the all-reference run produced (tests/golden/control_scenario.npz)."""
    g = np.load(os.path.join(golden_dir, "control_scenario.npz"))
    reads = P.scenario_reads()
    client = sim.SimClient(reads, int(g["chunk"]), int(g["n_polls"]), first_len=int(g["first_len"]))
    proc = SignalProcessor(Kit.create_from_version(str(g["kit"])))
    models = []
    for t in [str(t) for t in g["targets"]]:
        pth, yml = _write_model_files(tmp_path, t)
        models.append(Model(pth, get_config(yml), LOG, t))
    client.start_streaming_reads()
    ctl.serial_target(client, models, proc, str(tmp_path / f"ref_{mode}"), mode, float(g["threshold"]))
    with open(tmp_path / f"ref_{mode}.csv") as f:
        lines = [ln.rstrip("\n") for ln in f]
    assert lines[0] == str(g["header"])
    got = [ln.split(",", 1)[1].split(",") for ln in lines[1:]]
    want = [r.split(",") for r in g[f"rows_{mode}"]]
    assert len(got) == len(want)
    thr = float(g["threshold"])
    forgiven = 0
    for a, b in zip(got, want):
        assert a[:4] == b[:4], (a, b)                      # read id, channel, sig_length, models
        pa = np.array([float(x) for x in a[4].split(";")])
        pb = np.array([float(x) for x in b[4].split(";")])
        assert np.abs(pa - pb).max() < 1e-3
        assert a[5:7] == b[5:7]
        if a[7] != b[7]:
            assert np.abs(pb - thr).min() <= 1e-3, (a, b)
            forgiven += 1
    print(f"{len(got)} rows, {forgiven} decisions forgiven (reference p within 1e-3 of the threshold)")
    assert forgiven <= max(1, len(got) // 1000)
    assert sorted(map(tuple, g[f"unblocked_{mode}"])) == sorted(client.unblocked) or forgiven
    assert sorted(map(tuple, g[f"finished_{mode}"])) == sorted(client.finished) or forgiven


def test_mad_normalise_input_dtypes():
    """riser/preprocess.py:108-115 takes whatever dtype the client hands over.  Integers and integral float64 are
    the int16 path (float64 arithmetic, as numpy does for them); float32 stays float32 in numpy and here,
    bit for bit (the secondary input mode, SURVEY 8c); MAD == 0 gives the reference's int64 zeros."""
    proc = SignalProcessor(Kit.create_from_version("RNA002"))
    rng = np.random.default_rng(3)
    x16 = rng.normal(500, 60, 6000).astype(np.int16)
    x16[100:103] = 2000
    x16[0] = 1500
    x16[-1] = -900
    want = pp.mad_normalise(x16).astype(np.float32)
    for dt in (np.int16, np.int32, np.int64, np.float64):
        got = proc.mad_normalise(x16.astype(dt))
        assert got.dtype == np.float64 and np.array_equal(got.astype(np.float32), want), dt
    got = proc.mad_normalise(np.abs(x16).astype(np.uint16))
    assert np.array_equal(got.astype(np.float32), pp.mad_normalise(np.abs(x16)).astype(np.float32))
    # float32: numpy keeps float32 for the median, the MAD, the division and the smoothing
    for xf in (x16.astype(np.float32), (x16 * 0.1759 + 3.2).astype(np.float32)):
        got = proc.mad_normalise(xf)
        ref32 = _numpy_f32_normalise(xf)
        assert got.dtype == np.float32 and np.array_equal(got, ref32)
    # non-integral float64 takes the float32 route: inside the 1e-6 bar of the float64 result
    xd = x16 * 0.1759 + 3.2
    got = proc.mad_normalise(xd)
    ref64 = _numpy_f64_normalise(xd)
    ok = np.abs(ref64) < 3.4          # away from the outlier threshold the two precisions decide alike
    assert np.abs(got[ok] - ref64[ok]).max() <= 2e-6 * max(1.0, np.abs(ref64[ok]).max())
    # MAD == 0: int64 zeros for every input dtype (preprocess.py:122-124 through np.vectorize)
    for dt in (np.int16, np.float32, np.float64):
        z = proc.mad_normalise(np.full(5000, 7, dtype=dt))
        assert z.dtype == np.int64 and z.shape == (5000,) and not z.any()
    with pytest.raises(ValueError):
        proc.mad_normalise(np.zeros(0, dtype=np.float32))
    if refshim.available():                  # and against the reference itself when it can be imported
        rp = refshim.load().preprocess
        rproc = rp.SignalProcessor(rp.Kit.create_from_version("RNA002"))
        xf = (x16 * 0.1759 + 3.2).astype(np.float32)
        r = rproc.mad_normalise(xf)
        assert r.dtype == np.float32 and np.array_equal(r, proc.mad_normalise(xf))
        assert rproc.mad_normalise(np.full(5000, 7, dtype=np.float32)).dtype == np.int64


def _smooth(arr, lim=3.5):
    idx = np.asarray(np.abs(arr) > lim).nonzero()[0]
    for i in idx:
        if i == 0:
            arr[i] = arr[i + 1]
        elif i == len(arr) - 1:
            arr[i] = arr[i - 1]
        else:
            arr[i] = (arr[i - 1] + arr[i + 1]) / 2
            arr[i] = min(max(arr[i], -lim), lim)
    return arr


def _numpy_f32_normalise(x):
    """What numpy does with float32 input in preprocess.py:108-147: every step stays float32."""
    med = np.median(x)
    mad = np.median(np.abs(x - med))
    assert med.dtype == np.float32 and mad.dtype == np.float32
    return _smooth(((x - med) / (np.float32(1.4826) * mad)).astype(np.float32))


def _numpy_f64_normalise(x):
    med = np.median(x)
    mad = np.median(np.abs(x - med))
    return _smooth((x - med) / (1.4826 * mad))


def test_classify_batch_refuses_float_signal_and_converts_integers():
    """The batched path packs raw int16 samples; a client configured for calibrated (float) signal must not be
    misread silently (riser/client.py:47 uses the client's signal_dtype)."""
    from riser_b200 import BatchedClassifier
    from riser_b200.config import shipped_config
    model = Model(synth.state_dict(0), shipped_config(), LOG, "mRNA")
    clf = BatchedClassifier([model], SignalProcessor(Kit.create_from_version("RNA002")))
    reads = synth.raw_reads(3, 4, min_body=9000, max_body=12000)
    sigs, ids = [s for _, s in reads], [r for r, _ in reads]
    base = clf.classify_batch(sigs, ids, {}, 0.9, "deplete")
    wide = clf.classify_batch([s.astype(np.int32) for s in sigs], ids, {}, 0.9, "deplete")
    assert np.array_equal(base.decisions, wide.decisions) and np.array_equal(base.p_on, wide.p_on)
    with pytest.raises(TypeError):
        clf.classify_batch([s.astype(np.float32) for s in sigs], ids, {}, 0.9, "deplete")
    # empty batch through the public Model API (ADVICE): an empty [0, 2] tensor, no ZeroDivision / ValueError
    empty = model.classify_batch(torch.zeros(0, 4096, device=model.device), torch.zeros(0, dtype=torch.int32, device=model.device))
    assert tuple(empty.shape) == (0, 2) and model.launches(0, 4096) == 0
