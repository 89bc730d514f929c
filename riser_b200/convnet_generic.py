"""ConvNet shapes beyond the shipped one (riser/nets/cnn.py:8-65): ``depth`` > 1 (several Conv1d + ReLU before a
layer's pool, cnn.py:52-65), odd kernel sizes other than 3, any ``n_classes``, and the ``'gap'`` classifier
(Conv1d(C, n_classes, 1) + AdaptiveAvgPool1d, cnn.py:35-39).  ``riser_b200.Model`` builds this class when the
configuration is not the 12 x k3 depth-1 'gap_fc' two-class network the dedicated kernels of csrc/convnet.cu
are written for; the call surface (``classify``, ``classify_batch``) is the same.

It runs on the channel-last fp32 building blocks the ResNet variant uses (csrc/resnet_tc.cu, csrc/resnet.cu):
a k = 3 convolution whose shape the tensor-core kernel takes goes through ``riser_res_tc`` (tcgen05, fp16 hi + lo
operand planes, fp32 accumulation), any other through ``riser_conv1d_cl`` (fp32 CUDA cores); the unpadded
MaxPool1d(2, 2) is ``riser_maxpool1d_pad_cl``; 'gap_fc' and 'gap' are both ``riser_gap_linear_softmax`` -- a 1 x 1
convolution commutes with the average pool, so 'gap' is a linear layer on the pooled features with the conv's
weights.  The per-layer valid lengths of a ragged batch come from one ``riser_len_chain`` launch.  No CPU path.

Not taken: even kernel sizes (torch's padding='same' is asymmetric for them) and the 'fc' classifier, whose input
width is hard-coded to one configuration in the reference (cnn.py:24-29)."""
import numpy as np
import torch

from . import _lib
from .resnet import _Conv, _pad8


def check_supported(c):
    """Raise NotImplementedError for the ConvNet configurations riser_b200 does not implement (module docstring)."""
    if c.classifier not in ('gap_fc', 'gap'):
        raise NotImplementedError(f"classifier {c.classifier!r}: riser_b200 implements 'gap_fc' and 'gap' "
                                  "(the reference's 'fc' head is hard-coded to one input width, riser/nets/cnn.py:24-29)")
    if any(int(k) % 2 == 0 or int(k) < 1 for k in c.kernels[:int(c.n_layers)]):
        raise NotImplementedError("riser_b200 implements odd kernel sizes (padding='same' is asymmetric for even ones)")


class GenericConvNet:
    def __init__(self, sd, c, device, logger=None):
        self.device = device
        n = int(c.n_layers)
        depth = int(c.depth)
        self.n_classes = int(c.n_classes)
        channels = [int(x) for x in c.channels[:n]]
        kernels = [int(k) for k in c.kernels[:n]]
        check_supported(c)
        # expected keys and shapes: what ConvNet(config.cnn).load_state_dict enforces (cnn.py:13-41, 52-65)
        expected = {}
        cin = 1
        for i, (cout, k) in enumerate(zip(channels, kernels)):
            for d in range(depth):
                expected[f"layers.{i}.{2 * d}.weight"] = (cout, cin if d == 0 else cout, k)
                expected[f"layers.{i}.{2 * d}.bias"] = (cout,)
            cin = cout
        if c.classifier == 'gap_fc':
            head_w, head_b = "classifier.2.weight", "classifier.2.bias"
            expected[head_w] = (self.n_classes, channels[-1])
        else:
            head_w, head_b = "classifier.0.weight", "classifier.0.bias"
            expected[head_w] = (self.n_classes, channels[-1], 1)
        expected[head_b] = (self.n_classes,)
        missing = [k for k in expected if k not in sd]
        unexpected = [k for k in sd if k not in expected]
        if missing or unexpected:
            raise RuntimeError(f"Error(s) in loading state_dict for ConvNet: missing keys {missing}, "
                               f"unexpected keys {unexpected}")
        host = {}
        for k, shape in expected.items():
            t = torch.as_tensor(sd[k]).detach().to("cpu", torch.float32).contiguous()
            if tuple(t.shape) != shape:
                raise RuntimeError(f"size mismatch for {k}: checkpoint {tuple(t.shape)} vs model {shape}")
            host[k] = t
        max_smem = torch.cuda.get_device_properties(device).shared_memory_per_block_optin
        self.layers = []          # per layer: list of _Conv
        self.n_tc = self.n_cuda_core = 0
        for i, k in enumerate(kernels):
            convs = []
            for d in range(depth):
                first = (i == 0 and d == 0)
                cv = _Conv(host[f"layers.{i}.{2 * d}.weight"], host[f"layers.{i}.{2 * d}.bias"], 1, (k - 1) // 2, device,
                           pad_cin=not first)
                if not first and cv.build_tc(device, max_smem) is not None:
                    self.n_tc += 1
                else:
                    self.n_cuda_core += 1
                convs.append(cv)
            self.layers.append(convs)
        self.c_last_p = _pad8(channels[-1])
        fc = torch.zeros(self.n_classes, self.c_last_p)
        fc[:, :channels[-1]] = host[head_w].reshape(self.n_classes, channels[-1])
        self.fc_w = fc.contiguous().to(device)
        self.fc_b = host[head_b].contiguous().to(device)
        chain = []
        for convs in self.layers:
            chain += [(cv.k, 1, cv.pad) for cv in convs] + [(-1, 2, 0)]
        self.n_chain = len(chain)
        self.chain = torch.tensor(chain, dtype=torch.int32).contiguous().to(device)
        self.min_length = 1 << n         # shorter input leaves nothing for the last pool (the reference raises there)
        self._acts = {}
        if logger is not None:
            logger.debug('generic ConvNet: %d convs on tcgen05, %d on CUDA cores', self.n_tc, self.n_cuda_core)

    def _buf(self, key, *shape):
        t = self._acts.get((key,) + shape)
        if t is None:
            t = self._acts[(key,) + shape] = torch.empty(*shape, dtype=torch.float32, device=self.device)
        return t

    def _conv(self, cv, x, n_in, L, n_out):
        B = x.shape[0]
        out = self._buf(id(cv), B, L, cv.cout_p)
        lib, stream = _lib.lib(), _lib.stream_ptr()
        if cv.tc is not None:
            t = cv.tc
            _lib.check(lib.riser_res_tc(_lib.ptr(x), _lib.ptr(n_in), _lib.ptr(n_out), _lib.ptr(out), None, _lib.ptr(t["w"]),
                                        None, None, _lib.ptr(t["bias"]), None, t["inv"], 1.0, B, L, L, cv.cin_p, 0,
                                        cv.cout_p, t["n1"], 0, cv.k, 1, 1, stream), "riser_res_tc")
        else:
            _lib.check(lib.riser_conv1d_cl(_lib.ptr(x), _lib.ptr(n_in), _lib.ptr(cv.w), _lib.ptr(cv.b), None, _lib.ptr(out),
                                           _lib.ptr(n_out), B, L, L, cv.cin_p, cv.cout_p, cv.k, 1, cv.pad, 1, stream),
                       "riser_conv1d_cl")
        return out

    def classify_batch(self, x, lens, max_len=None, probs=None, **_unused):
        """x: fp32 [B, ld] normalised signals on the device, lens int32 [B] -> probs fp32 [B, n_classes]
        (NaN rows for reads too short for the last pool).  No synchronisation."""
        B = x.shape[0]
        if probs is None:
            probs = torch.empty(B, self.n_classes, dtype=torch.float32, device=self.device)
        if B == 0:
            return probs
        L = int(max_len if max_len is not None else x.shape[1])
        lens = lens.to(torch.int32)
        n_all = self._buf_i32(B)
        lib, stream = _lib.lib(), _lib.stream_ptr()
        _lib.check(lib.riser_len_chain(_lib.ptr(lens), B, _lib.ptr(self.chain), self.n_chain, _lib.ptr(n_all), stream),
                   "riser_len_chain")
        h = x[:, :L].contiguous().view(B, L, 1)
        n, j = lens, 0
        for convs in self.layers:
            for cv in convs:
                h = self._conv(cv, h, n, L, n_all[j])
                n = n_all[j]
                j += 1
            Lp = max(1, L // 2)
            pooled = self._buf(("pool", id(convs[-1])), B, Lp, convs[-1].cout_p)
            _lib.check(lib.riser_maxpool1d_pad_cl(_lib.ptr(h), _lib.ptr(n), _lib.ptr(pooled), _lib.ptr(n_all[j]), B, L, Lp,
                                                  convs[-1].cout_p, 0, stream), "riser_maxpool1d_pad_cl")
            h, n, L = pooled, n_all[j], Lp
            j += 1
        _lib.check(lib.riser_gap_linear_softmax(_lib.ptr(h), _lib.ptr(n), _lib.ptr(self.fc_w), _lib.ptr(self.fc_b),
                                                _lib.ptr(probs), B, L, self.c_last_p, self.n_classes, stream),
                   "riser_gap_linear_softmax")
        return probs

    def _buf_i32(self, B):
        t = self._acts.get(("len", B))
        if t is None:
            t = self._acts[("len", B)] = torch.empty(self.n_chain, B, dtype=torch.int32, device=self.device)
        return t

    def launches(self, B):
        return 0 if B <= 0 else 1 + self.n_chain + 1

    def classify(self, signal):
        signal = np.asarray(signal)
        n = signal.shape[0]
        x = torch.from_numpy(signal).to(self.device, dtype=torch.float).view(1, n)
        lens = torch.tensor([n], dtype=torch.int32, device=self.device)
        return self.classify_batch(x, lens, max_len=n)[0]
