"""Input-pipeline edge (SURVEY.md 8 f3): uint8 batches normalised on the device are BIT-identical to the reference's host
pipeline - TorchMeanStdNormalize (ToTensor: uint8 HWC -> float CHW / 255; Normalize: sub_(mean).div_(std);
reference SimpleAICV/classification/common.py:228-248) followed by ClassificationCollater's stack + permute
(:645-665) - for vector-friendly and odd image sizes, directly and through the prefetcher."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def _host_pipeline(images_u8, mean, std):
    """What the reference computes on the host for a list of uint8 HWC images."""
    out = []
    for img in images_u8:
        t = torch.from_numpy(img).permute(2, 0, 1).contiguous().to(torch.float32).div(255)     # transforms.ToTensor
        m = torch.tensor(mean, dtype=torch.float32).view(3, 1, 1)
        s = torch.tensor(std, dtype=torch.float32).view(3, 1, 1)
        t = t.sub_(m).div_(s)                                                                   # transforms.Normalize
        out.append(t.permute(1, 2, 0).numpy())                                                  # back to HWC (common.py:243)
    batch = torch.from_numpy(np.array(out).astype(np.float32)).float().permute(0, 3, 1, 2)      # collater
    return batch


@pytest.mark.parametrize('n,h,w', [(4, 224, 224), (3, 37, 41), (2, 32, 32), (1, 5, 7)])
@pytest.mark.parametrize('mean,std', [(MEAN, STD), ((0., 0., 0.), (1., 1., 1.))])
def test_device_normalize_is_bit_identical_to_the_host_pipeline(n, h, w, mean, std):
    from simpleaicv_pytorch_training_examples_b200.classification.common import DeviceNormalize
    rng = np.random.default_rng(n * 1000 + h)
    imgs = [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for _ in range(n)]
    ref = _host_pipeline(imgs, mean, std)
    got = DeviceNormalize(mean, std)(torch.from_numpy(np.stack(imgs)).cuda())
    assert got.shape == (n, 3, h, w) and got.dtype == torch.float32 and got.is_contiguous()
    assert torch.equal(got.cpu(), ref.contiguous())


def test_prefetcher_moves_uint8_and_normalises_on_the_copy_stream():
    from simpleaicv_pytorch_training_examples_b200.classification.common import DeviceNormalize, Uint8ClassificationCollater
    from simpleaicv_pytorch_training_examples_b200.tools.utils import CudaPrefetcher
    rng = np.random.default_rng(7)
    collate = Uint8ClassificationCollater()
    samples = [[{'image': rng.integers(0, 256, size=(64, 64, 3), dtype=np.uint8), 'label': int(rng.integers(0, 10))}
                for _ in range(8)] for _ in range(5)]
    loader = [collate(s) for s in samples]
    assert loader[0]['image'].dtype == torch.uint8 and loader[0]['image'].is_pinned() and loader[0]['label'].dtype == torch.int64
    seen = 0
    for batch, raw in zip(CudaPrefetcher(loader, normalize=(MEAN, STD)), samples):
        ref = _host_pipeline([s['image'] for s in raw], MEAN, STD)
        assert batch['image'].dtype == torch.float32 and tuple(batch['image'].shape) == (8, 3, 64, 64)
        assert torch.equal(batch['image'].cpu(), ref.contiguous())
        assert batch['label'].tolist() == [s['label'] for s in raw]
        seen += 1
    assert seen == 5
    with pytest.raises(RuntimeError):
        DeviceNormalize(MEAN, STD)(loader[0]['image'])     # CPU tensor: no host fallback
