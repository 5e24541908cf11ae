"""fact_gather_windows and create_device_input on the GPU: the kernel against slicing, the device producer against
create_input, and training fed by either."""
import ctypes

import numpy as np
import pytest
import torch

from mint_b200 import device_inputs, inputs
from mint_b200 import lib as L
from tests.golden import make_input_stream_golden as G

pytestmark = pytest.mark.gpu

FACT_WINDOW = dict(motion_dim=225, audio_dim=35, motion_len=120, target_shift=120, target_len=20, audio_len=240)
ODD_WINDOW = dict(motion_dim=7, audio_dim=3, motion_len=5, target_shift=4, target_len=3, audio_len=9)


def _gather(fact_lib, motion, audio, m_rows, a_rows, w):
    b = m_rows.numel()
    outs = [torch.full((b, w["motion_len"], w["motion_dim"]), float("nan"), device=motion.device),
            torch.full((b, w["target_len"], w["motion_dim"]), float("nan"), device=motion.device),
            torch.full((b, w["audio_len"], w["audio_dim"]), float("nan"), device=motion.device)]
    L.check(fact_lib.fact_gather_windows(motion.data_ptr(), w["motion_dim"], audio.data_ptr(), w["audio_dim"],
                                         m_rows.data_ptr(), a_rows.data_ptr(), b, w["motion_len"], w["target_shift"],
                                         w["target_len"], w["audio_len"], *(o.data_ptr() for o in outs),
                                         torch.cuda.current_stream().cuda_stream), "fact_gather_windows")
    return outs


@pytest.mark.parametrize("batch", [1, 3, 32, 128, 256])
@pytest.mark.parametrize("window", ["fact", "odd"])
def test_gather_windows_equals_slicing(cuda, fact_lib, batch, window):
    w = FACT_WINDOW if window == "fact" else ODD_WINDOW
    g = torch.Generator(device="cpu").manual_seed(batch)
    rows_m, rows_a = 3001, 2777
    motion = torch.randn(rows_m, w["motion_dim"], generator=g).to(cuda)
    audio = torch.randn(rows_a, w["audio_dim"], generator=g).to(cuda)
    last_m = rows_m - max(w["motion_len"], w["target_shift"] + w["target_len"])
    last_a = rows_a - w["audio_len"]
    m_rows = torch.randint(0, last_m + 1, (batch,), generator=g)
    a_rows = torch.randint(0, last_a + 1, (batch,), generator=g)
    m_rows[0], a_rows[0] = last_m, last_a                    # the last valid starts
    if batch > 1:
        m_rows[-1], a_rows[-1] = 0, 0                        # and the first
    outs = _gather(fact_lib, motion, audio, m_rows.to(cuda), a_rows.to(cuda), w)
    torch.cuda.synchronize()
    ts = w["target_shift"]
    want = [torch.stack([motion[r:r + w["motion_len"]] for r in m_rows.tolist()]),
            torch.stack([motion[r + ts:r + ts + w["target_len"]] for r in m_rows.tolist()]),
            torch.stack([audio[r:r + w["audio_len"]] for r in a_rows.tolist()])]
    for o, e in zip(outs, want):
        assert torch.equal(o, e)


def test_gather_windows_rejects_bad_arguments(cuda, fact_lib):
    w = FACT_WINDOW
    motion = torch.zeros(400, 225, device=cuda)
    audio = torch.zeros(400, 35, device=cuda)
    rows = torch.zeros(2, dtype=torch.int64, device=cuda)
    outs = [torch.empty(2, 120, 225, device=cuda), torch.empty(2, 20, 225, device=cuda),
            torch.empty(2, 240, 35, device=cuda)]
    st = torch.cuda.current_stream().cuda_stream
    good = [motion.data_ptr(), 225, audio.data_ptr(), 35, rows.data_ptr(), rows.data_ptr(), 2, w["motion_len"],
            w["target_shift"], w["target_len"], w["audio_len"], *(o.data_ptr() for o in outs), st]
    assert fact_lib.fact_gather_windows(*good) == 0
    for i, bad in ((6, 0), (6, 70000), (1, 0), (3, -1), (7, 0), (8, -1), (9, 0), (10, 0), (0, None), (5, None),
                   (12, None)):
        args = list(good)
        args[i] = bad
        assert fact_lib.fact_gather_windows(*args) == -1, (i, bad)
        assert b"fact_gather_windows" in fact_lib.fact_last_error(), (i, bad)
    torch.cuda.synchronize()


@pytest.fixture(scope="module")
def layouts(tmp_path_factory):
    out = {}
    for name, counts in (("one", [7]), ("several", [40, 50, 40])):
        root = tmp_path_factory.mktemp(name)
        out[name] = (G.write_layout(str(root), counts, (240, 300), seed=len(counts)), sum(counts))
    return out


@pytest.mark.parametrize("name,batch_size,seed,per_block", [("one", 3, 4, 3), ("several", 32, 3, 4),
                                                             ("several", 1, 9, 64)])
def test_create_device_input_equals_create_input(cuda, fact_lib, layouts, name, batch_size, seed, per_block):
    """Bit for bit over more than two epochs, across row-table blocks, with some steps drawn on another stream."""
    files, records = layouts[name]
    cfg = G.configs(files, batch_size)
    host = inputs.create_input(cfg["train_config"], cfg["train_dataset"], is_training=True, seed=seed)
    dev = device_inputs.create_device_input(cfg["train_config"], cfg["train_dataset"], cuda, seed=seed,
                                            steps_per_block=per_block)
    side = torch.cuda.Stream()
    got = []
    for s in range(-(-2 * records // batch_size) + 2):
        if s % 3 == 2:
            with torch.cuda.stream(side):
                got.append(next(dev))
        else:
            got.append(next(dev))
    torch.cuda.synchronize()
    for s, b in enumerate(got):
        want = next(host)
        assert list(b) == list(want), s
        for k, v in want.items():
            if isinstance(v, np.ndarray):
                t = torch.from_numpy(v)
                assert b[k].device.type == "cuda" and b[k].dtype == t.dtype and torch.equal(b[k].cpu(), t), (s, k)
            else:
                assert b[k] == v, (s, k)


def test_training_fed_by_either_producer(cuda, fact_lib, layouts):
    """Three SingleTaskTrainer steps per producer from identical weights.  The batches are bit-identical and so is the
    first loss; the backward's bulk gradient reductions are unordered (tests/test_train_gpu.py), so later losses and
    the weights agree to that reduction order only."""
    from mint_b200.fact_model import FACTModel
    from mint_b200.optim import Adam
    from mint_b200.trainer import SingleTaskTrainer
    from tests.helpers import make_config
    files, _ = layouts["several"]
    cfg = G.configs(files, 4)
    keys = ("motion_input", "audio_input", "target")
    feeds = {"host": inputs.create_input(cfg["train_config"], cfg["train_dataset"], is_training=True, seed=1),
             "device": device_inputs.create_device_input(cfg["train_config"], cfg["train_dataset"], cuda, seed=1)}
    seen, losses, weights = {}, {}, {}
    w0 = None
    for name, feed in feeds.items():
        model = FACTModel(make_config(d=64, heads=4, ff=128, layers=(1, 1, 2)), is_training=True, mode="bf16", seed=3)
        w0 = model.flat_parameters.clone() if w0 is None else w0
        assert torch.equal(model.flat_parameters, w0)
        batches = [{k: b[k] for k in keys} for b in (next(feed) for _ in range(3))]
        seen[name] = batches
        trainer = SingleTaskTrainer(iter(batches), "target", model, optimizer=Adam(model, learning_rate=1e-3))
        losses[name] = [float(trainer.train_step(b)) for b in batches]
        weights[name] = model.flat_parameters.clone()
    for hb, db in zip(seen["host"], seen["device"]):
        for k in keys:
            assert torch.equal(torch.as_tensor(hb[k]), db[k].cpu()), k
    assert losses["host"][0] == losses["device"][0]
    for a, b in zip(losses["host"], losses["device"]):
        assert abs(a - b) <= 1e-5 * abs(a), losses
    moved = float((weights["host"] - w0).double().norm())
    assert moved > 0
    assert float((weights["host"] - weights["device"]).double().norm()) <= 1e-3 * moved
