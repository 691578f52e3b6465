"""The batched two-stage path as one call: `pipeline(imgs) -> (masks, boxes, logits)` (SURVEY.md §8b).

Replaces the reference's per-image loop (分类/test.py:122-134 calling roi.py:12-51 inside the Dataset, then
test.py:81-86) with one engine program per micro-batch: no host round trip between the UNet and GoogLeNet."""
import torch

from .lower import PipelineRunner


class TwoStagePipeline:
    def __init__(self, unet, classifier, micro_batch=64, padding=30, cls_batch=256):
        """unet: nets.UNetTaskAligWeight (or a reference-format state_dict); classifier: GoogLeNetClassifier
        (or its state_dict).  Both must live on the same CUDA device."""
        usd = unet if isinstance(unet, dict) else unet.state_dict()
        gsd = classifier if isinstance(classifier, dict) else classifier.state_dict()
        dev = next(iter(usd.values())).device if isinstance(unet, dict) else unet.outc.weight.device
        if torch.device(dev).type != "cuda":
            dev = torch.device("cuda", torch.cuda.current_device())
        self.runner = PipelineRunner(usd, gsd, dev, micro_batch=micro_batch, padding=padding, cls_batch=cls_batch)

    @torch.no_grad()
    def __call__(self, imgs, return_logits=False, return_cam=False, return_source=False):
        """imgs: float [B,3,224,224] on the pipeline's device, or uint8 HWC sources [B,Hs,Ws,3] of any size (resized
        on the device like the reference's CDDataAugmentation.transform: PIL bilinear + to_tensor), or a list of uint8
        [H,W,3] images of different sizes (CUDA tensors or numpy arrays; run as ragged batches, util/ragged.py) ->
        (masks uint8 [B,224,224], boxes int32 [B,4] = (x0,y0,x1,y1), class logits float32 [B,6]), followed by the
        segmentation logits if return_logits and by the Grad-CAM map of the predicted class (float32 [B,224,224], in
        the 224x224 frame, inside each image's box) if return_cam, and by a SourceFrame(masks, boxes, cam_maps) of the
        same outputs at each source image's own size if return_source (uint8 sources only; lists of per-image tensors
        for a list of images; cam_maps is None without return_cam)."""
        return self.runner(imgs, return_logits=return_logits, return_cam=return_cam, return_source=return_source)

    def predict(self, imgs):
        """argmax(softmax(logits)) as 分类/test.py:86 (softmax is monotone, so argmax of the logits)."""
        return torch.argmax(self(imgs)[2], dim=1)
