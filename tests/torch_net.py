"""The policy/value network in torch, from the folded C-ABI weight vector (the layout of
cb200_trainer_set_weights): an evaluator that lives on the GPU, for driving the analysis' device
forms. Rows [k, 70] float32 CUDA tensor -> (eval [k], probs [k, 96]), contiguous float32 on the
rows' device. fp32 math in torch's own kernels, so its answers are not bit-identical to the
engine's network kernels; the tests that use it compare the engine with itself."""
import numpy as np

DIMS = [70] + [100] * 12 + [97]


def torch_network(flat_weights, device):
    import torch
    flat = np.ascontiguousarray(flat_weights, np.float32)
    layers, off = [], 0
    for k, n in zip(DIMS[:-1], DIMS[1:]):
        w = torch.from_numpy(flat[off:off + k * n].reshape(k, n).copy()).to(device)
        off += k * n
        b = torch.from_numpy(flat[off:off + n].copy()).to(device)
        off += n
        layers.append((w, b))

    @torch.no_grad()
    def evaluate(rows):
        h = rows
        for i, (w, b) in enumerate(layers):
            h = torch.addmm(b, h, w)
            if i < len(layers) - 1:
                h = torch.relu(h)
        return torch.tanh(h[:, 0]).contiguous(), torch.softmax(h[:, 1:], dim=1).contiguous()
    return evaluate
