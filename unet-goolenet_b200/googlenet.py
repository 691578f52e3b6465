"""Drop-in shell of the reference's stage-2 classifier (分类/test.py:64-73 == 分类/ROI_main.py:86-95).

`GoogLeNetClassifier(num_classes=6)` exposes the same `.googlenet` child with torchvision's parameter names
(344 state_dict tensors, no aux heads), so `load_state_dict(torch.load(p)['net'])` works unchanged; forward runs
on the ugnet engine.  The reference builds torchvision's googlenet(pretrained=True), which implies
transform_input=True and drops the aux heads; there is no network here, so the structurally identical
`googlenet(weights=None, aux_logits=False, transform_input=True, init_weights=False)` is constructed instead
(pass `pretrained_state` to start from an ImageNet state_dict you have on disk)."""
import torch
import torch.nn as nn


class GoogLeNetClassifier(nn.Module):
    def __init__(self, num_classes=6, pretrained_state=None):
        super().__init__()
        import torchvision
        net = torchvision.models.googlenet(weights=None, aux_logits=False, transform_input=True, init_weights=False)
        if pretrained_state is not None:
            net.load_state_dict({k: v for k, v in pretrained_state.items() if not k.startswith("aux")})
        net.fc = nn.Linear(net.fc.in_features, num_classes)
        self.googlenet = net
        self._runner = None
        self._register_load_state_dict_pre_hook(self._drop_runner)

    def _drop_runner(self, *args, **kwargs):
        self._runner = None

    def invalidate(self):
        """Forget the packed engine copy of the weights (it is rebuilt on the next forward)."""
        self._runner = None

    def _fingerprint(self):
        # (storage address, in-place version counter) of every parameter / buffer: changes on load_state_dict, .to(),
        # optimizer steps, p.copy_() / p.mul_() under no_grad, and on assigning a new Parameter or submodule.  Writes
        # through `p.data` bypass the version counter: call invalidate() after those.
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_runner"] = None          # the engine handle / device workspaces are per process, never pickled
        state.pop("_runner_key", None)
        return state

    def __deepcopy__(self, memo):
        import copy
        runner, self._runner = self._runner, None
        try:
            cls = self.__class__
            new = cls.__new__(cls)
            memo[id(self)] = new
            new.__dict__ = copy.deepcopy({k: v for k, v in self.__dict__.items() if k != "_runner_key"}, memo)
        finally:
            self._runner = runner
        return new

    def _apply(self, fn, *args, **kwargs):
        self._runner = None
        return super()._apply(fn, *args, **kwargs)

    def runner(self):
        key = self._fingerprint()
        if self._runner is not None and getattr(self, "_runner_key", None) != key:
            self._runner = None          # weights were edited in place since the last pack
        if self._runner is None:
            from .lower import GoogLeNetRunner
            dev = self.googlenet.fc.weight.device
            if dev.type != "cuda":
                raise RuntimeError("GoogLeNetClassifier runs on the ugnet CUDA engine only: call .to('cuda')")
            self._runner = GoogLeNetRunner(self.state_dict(), dev)
            self._runner_key = key
        return self._runner

    def forward(self, x):
        if self.training:
            raise RuntimeError("the ugnet engine is inference-only: call model.eval() (test.py:75)")
        return self.runner().forward(x)

    def grad_cam(self, x, classes=None):
        """Grad-CAM at `googlenet.inception5b`, the engine form of pytorch-grad-cam's
        `GradCAM(model, target_layers=[model.googlenet.inception5b])(x, targets)` followed by its scale_cam_image:
        x float [B,3,224,224] in [0,1] -> (cam_map f32 [B,224,224] in [0,1], cam f32 [B,7,7]), both in the crop frame.
        classes: int [B] target classes, or None for each image's predicted class (argmax of the logits).
        GoogLeNet's head is avgpool -> fc, so the Grad-CAM weights are fc.weight[c] / 49 and no backward pass runs."""
        if self.training:
            raise RuntimeError("the ugnet engine is inference-only: call model.eval() (test.py:75)")
        return self.runner().grad_cam(x, classes)
