"""The whole-model C entry (include/svnet_b200.h: svnet_model_create / _forward / _destroy) behind a Python callable --
what a C or C++ host would do with the library, spelled out: build the handle from a checkpoint's tensors once, then
`forward` with caller-owned scratch.  Covered: SV_DGCNN_CLS, binary (k = 20 / 40) or full precision (k = 20), and
SV_DGCNN_PSEG, binary or full precision (k = 20 / 40; `native(batch, label_one_hot)` -> (B, parts, N)); 64 <= N <= 4096.

    native = svnet_b200.NativeModel("SV_DGCNN_CLS", checkpoint["state_dict"], k=20, binary=True, num_class=40)
    logits = native(batch)                     # (B, 3, N) float32 CUDA -> (B, num_class); bit-identical to the nn.Module

The nn.Module classes remain the drop-in for the reference's Python code; this class exists for hosts without Python
model code and as the executable documentation of the C entry.
"""
import torch

from . import _native as nv


class NativeModel:
    def __init__(self, kind, state_dict, k, binary, num_class, device=None):
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        with torch.cuda.device(dev):
            sd = {n: t.to(dev) for n, t in state_dict.items() if torch.is_tensor(t) and t.dtype == torch.float32}
            self._h = nv.model_create(kind, k, binary, num_class, sd)
        self.device, self.num_class, self.kind, self.binary = dev, num_class, kind, bool(binary)
        self._ws = {}          # scratch per batch shape, kept for the handle's lifetime (a captured CUDA graph may hold its address)

    def __call__(self, x, label=None):
        if not x.is_cuda:
            raise RuntimeError("NativeModel needs a CUDA tensor (there is no CPU path)")
        B, _, N = x.shape
        if self.kind == "SV_DGCNN_PSEG":
            if label is None:
                raise TypeError("SV_DGCNN_PSEG needs the one-hot object label (B, 16)")
            with torch.cuda.device(x.device):
                key = (B, N)
                if key not in self._ws:
                    nbytes = nv.model_seg_workspace_bytes(self._h, B, N)
                    if nbytes == 0:
                        raise ValueError("shape (B=%d, N=%d) is not covered by svnet_model_forward_seg (64 <= N <= 4096; a full-precision "
                                         "model also needs the tensor-core linear for its head's conv8)" % (B, N))
                    self._ws[key] = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
                logits = torch.empty((B, self.num_class, N), dtype=torch.float32, device=x.device)
                nv.model_forward_seg(self._h, x.contiguous(), label.reshape(B, -1).contiguous().float(), logits, self._ws[key])
                if self.binary:       # kernels behind the one call (per sub-batch: trunk 24, conv5 / conv6 branch 18, head 11, ...)
                    nv.LAUNCHES[0] += 60 * self._sub_batches(B, N) - 1
                # the full-precision model's call is counted as one launch: its kernel count is not derived here
            return logits
        with torch.cuda.device(x.device):
            key = (B, N)
            if key not in self._ws:
                nbytes = nv.model_workspace_bytes(self._h, B, N)
                if nbytes == 0:
                    raise ValueError("shape (B=%d, N=%d) is not covered by svnet_model_forward (64 <= N <= 4096)" % (B, N))
                self._ws[key] = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            logits = torch.empty((B, self.num_class), dtype=torch.float32, device=x.device)
            nv.model_forward(self._h, x.contiguous(), logits, self._ws[key])
            nv.LAUNCHES[0] += (33 if self.binary else 38) * self._sub_batches(B, N) - 1     # kernels behind the one call
        return logits

    @staticmethod
    def _sub_batches(B, N):
        """svnet_model_forward runs a batch as up to four sub-batches of >= 16 384 points (csrc/model.cu: split_count)."""
        return max(1, min(4, (B * N) // 16384, B))

    def close(self):
        if getattr(self, "_h", None) is not None:
            nv.model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
