"""train.py --image-size: the tiny model trains at any image size; the other models refuse it (CPU)."""
import pytest


@pytest.mark.parametrize("model", ["mnist", "fashion", "cifar10", "cifar2", "svhn", "emotion"])
def test_image_size_is_refused_for_fixed_size_heads(model):
    import cnn_with_pde_b200.train as train
    with pytest.raises(ValueError, match="only the tiny model takes other image sizes"):
        train.run(model, 2, 1, 0, quiet=True, image_size=224)


def test_image_size_must_be_positive():
    import cnn_with_pde_b200.train as train
    with pytest.raises(ValueError, match="must be positive"):
        train.run("tiny", 2, 1, 0, quiet=True, image_size=0)


def test_image_size_flag_reaches_run(monkeypatch):
    import cnn_with_pde_b200.train as train
    seen = {}
    monkeypatch.setattr(train, "run", lambda *a, **k: seen.update(k) or {"img_per_s": 0.0, "n_gpus": 1, "ms_per_step": 0.0})
    train.main(["--model", "tiny", "--image-size", "224", "--steps", "1"])
    assert seen["image_size"] == 224
