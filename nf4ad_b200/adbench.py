"""`ADBenchFlow`: the sklearn/ADBench-style wrapper nf4ad puts around a flow
(`/root/reference/src/nf4ad/adbench_wrapper.py:296-449`), on the B200 path.

Same constructor arguments, `fit(X_train, y_train=None)`, `predict_score(X_test)` (anomaly score =
-log_prob) and `predict(X_test, threshold=None)` contract; the reference's own class also works unchanged
on top of the drop-in (it only calls `flow.to / parameters / train / eval / log_prob`).  What this
mirror adds is the B200-specific plumbing around the same semantics:

  * `predict_score` streams pinned host rows in chunks whose H2D copies overlap the fused launch chain
    (`ShardedScorer.predict_score_host`) instead of one blocking copy of the whole test set
    (`adbench_wrapper.py:419`), and shards rows over the GPUs of a `torch.distributed` job;
  * `fit` keeps the training set on the device (one H2D copy), draws the shuffled mini-batches there, reads
    the loss back once per epoch instead of once per step (`adbench_wrapper.py:392` syncs every step), and
    replays the whole step (forward, backward kernels, Adam) as ONE CUDA graph per batch shape after a few
    eager steps (`DataParallelTrainer`); under `torch.distributed` it runs data parallel with one gradient
    all-reduce per step.
"""
from typing import Optional

import numpy as np
import torch

from .optim import FusedAdam
from .parallel import DataParallelTrainer, ShardedScorer, rank_batches, shared_permutation


class ADBenchFlow:
    def __init__(self, flow_model, batch_size: int = 32, epochs: int = 50, lr: float = 1e-3,
                 device: Optional[str] = None, gradient_clip: Optional[float] = None, verbose: bool = True):
        self.flow_model = flow_model
        self.batch_size, self.epochs, self.lr = batch_size, epochs, lr
        self.gradient_clip, self.verbose = gradient_clip, verbose
        if device is None:
            if not torch.cuda.is_available():
                raise RuntimeError("nf4ad_b200.ADBenchFlow needs a CUDA (sm_100a) device; there is no CPU path")
            self.device = torch.device("cuda", torch.cuda.current_device())
        else:
            self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError(f"nf4ad_b200.ADBenchFlow runs on CUDA only, got device={self.device}")
        self.flow_model.to(self.device)
        self.training_losses = []

    def fit(self, X_train: np.ndarray, y_train: Optional[np.ndarray] = None):
        """Minimise -mean log_prob with Adam over shuffled mini-batches (adbench_wrapper.py:347-404)."""
        with torch.cuda.device(self.device):
            return self._fit(X_train)

    def _fit(self, X_train):
        X = torch.as_tensor(np.asarray(X_train), dtype=torch.float32)
        if self.verbose:
            print(f"Training Flow model on {len(X)} samples...")
            print(f"Input shape: {X.shape}")
            print(f"Device: {self.device}")
        X = X.to(self.device)
        n = X.shape[0]
        opt = FusedAdam(self.flow_model.parameters(), lr=self.lr)   # torch.optim.Adam's update in one launch per 32 tensors; device-side step counter: the step replays as a CUDA graph
        trainer = DataParallelTrainer(self.flow_model, opt, gradient_clip=self.gradient_clip)
        trainer.broadcast_parameters()
        self.flow_model.train()
        self.training_losses = []
        gen = torch.Generator(device=self.device)
        gen.manual_seed(int(torch.initial_seed()) & 0x7FFFFFFF)
        for epoch in range(self.epochs):
            # data parallel: every rank walks the same global batches and trains on its shard of each
            perm = shared_permutation(n, self.device, gen, group=trainer.group)
            total = torch.zeros((), device=self.device)
            steps = 0
            for idx in rank_batches(perm, self.batch_size, trainer.rank, trainer.world):
                total += trainer.step(X.index_select(0, idx))
                steps += 1
            epoch_loss = float(total.cpu()) / max(steps, 1)      # one device->host sync per epoch
            self.training_losses.append(epoch_loss)
            if self.verbose and (epoch + 1) % 10 == 0:
                print(f"Epoch {epoch + 1}/{self.epochs}, Loss: {epoch_loss:.4f}")
        if self.verbose and self.training_losses:
            print(f"Training completed. Final loss: {self.training_losses[-1]:.4f}")
        return self

    def predict_score(self, X_test: np.ndarray) -> np.ndarray:
        """Anomaly score = -log_prob, per sample (adbench_wrapper.py:406-433)."""
        with torch.cuda.device(self.device):
            return self._predict_score(X_test)

    def _predict_score(self, X_test):
        X = torch.as_tensor(np.asarray(X_test), dtype=torch.float32)
        self.flow_model.eval()
        scorer = self.__dict__.get("_scorer")
        if scorer is None or scorer.flow is not self.flow_model:
            scorer = self._scorer = ShardedScorer(self.flow_model)     # keeps its pinned staging ring between calls
        if scorer.world > 1:
            return scorer.predict_score(X).numpy()
        # pageable rows go through the scorer's pinned staging ring (host thread pool), chunk by chunk, overlapped with
        # the PCIe copy and the compute -- no whole-array pin_memory() copy
        return scorer.predict_score_host(X).numpy()

    def score_gradients(self, X_test: np.ndarray, chunk_rows: int = 65536) -> np.ndarray:
        """Gradient of the anomaly score with respect to the input, -d log p(x) / dx, shape of X_test: which features make
        a sample anomalous.  Rows go to the device `chunk_rows` at a time (`Flow.log_prob_and_grad`)."""
        with torch.cuda.device(self.device):
            X = torch.as_tensor(np.asarray(X_test), dtype=torch.float32)
            self.flow_model.eval()
            out = np.empty(tuple(X.shape), dtype=np.float32)
            for i in range(0, X.shape[0], chunk_rows):
                _, g = self.flow_model.log_prob_and_grad(X[i:i + chunk_rows].to(self.device))
                out[i:i + chunk_rows] = (-g).cpu().numpy()
            return out

    def predict(self, X_test: np.ndarray, threshold: Optional[float] = None) -> np.ndarray:
        """1 = anomaly.  Default threshold: median score (adbench_wrapper.py:435-449)."""
        scores = self.predict_score(X_test)
        if threshold is None:
            threshold = np.median(scores)
        return (scores > threshold).astype(int)
