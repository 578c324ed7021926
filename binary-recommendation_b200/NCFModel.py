"""NCFModel -- drop-in mirror of the reference's serve-only class (src/models/NCFModel.py): the NeuMF network of the
script trainers/NFC_plain.py (latent 10, Dense 100-50-10 sigmoid, BCE, head [pred_mf, pred_mlp]; :109-155) restored
from a checkpoint and queried per user over ALL product ids of its training file.

The reference's predictForUser (:42-51) runs model.predict over one (customer, product) frame, drops predictions
>= 1.0, sorts the rest descending and returns {product: '%.9f' % score} for the best numberOfItem.  Here the frame is
the forward kernels of csrc/neumf.cu over the catalog (inference mode) and the selection a device top-k
(predictions >= 1.0 masked out first); several users go through predictForUsers in one pass.
"""
import numpy as np
import torch

from . import hotpath as H
from .NeuMFModel import NeuMFNet
from .RModel import RModel

SCRIPT_SPEC = dict(numFactor=10, hidden=(100, 50, 10), act="sigmoid", loss="bce", learning_rate=0.005,
                   head_order="mf_h3")                                  # NFC_plain.py:109-155


class NCFModel(RModel):
    def __init__(self, workDir=None, trainData=None):
        super().__init__('NCFModel', workDir)
        self._productIds: list = []
        self._customerIds: list = []
        # the reference hard-codes an SMB path (NCFModel.py:13) and loads it in the constructor; here the file is
        # optional at construction (a checkpoint carries both id lists) and any local CSV / .brkc cache is accepted
        self.trainData = trainData
        if trainData is not None:
            self.loadTrainData()

    @property
    def customerIds(self) -> list:
        return self._customerIds

    @customerIds.setter
    def customerIds(self, ids: list):
        self._customerIds = ids

    @property
    def productIds(self) -> list:
        return self._productIds

    @productIds.setter
    def productIds(self, ids: list):
        self._productIds = ids

    def compileModel(self, distributedConfig, numUser: int, numItem: int, numFactor: int = 10):
        spec = dict(SCRIPT_SPEC); spec["numFactor"] = numFactor
        self.model = NeuMFNet(numUser, numItem, dropout=0.0, seed=self.seed, **spec)
        return self.model

    def getPredictDataFrame(self, customerId):
        """NCFModel.py:32-35: one row per product id, the customer repeated."""
        return {'PRODUCT_ID': list(self.productIds), 'CUSTOMER_ID': [customerId] * len(self.productIds)}

    def checkpointMeta(self) -> dict:
        return {"model": self.modelName, "numUser": self.model.numUser, "numItem": self.model.numItem,
                "numFactor": self.model.E, "productIds": [int(x) for x in self.productIds],
                "customerIds": [int(x) for x in self.customerIds]}

    def buildFromMeta(self, meta: dict):
        self.compileModel(None, meta["numUser"], meta["numItem"], meta.get("numFactor", 10))
        if not self.productIds:
            self.productIds = list(meta.get("productIds", []))
        if not self.customerIds:
            self.customerIds = list(meta.get("customerIds", []))

    def predictForUsers(self, customerIds, numberOfItem=5):
        """[{product: '%.9f' % score, ...} per customer], best first (dicts keep insertion order)."""
        customerIds = [int(c) for c in customerIds]
        if self.model is None:
            raise RuntimeError("NCFModel: restoreFromLatestCheckPoint() or compileModel() first")
        bad = [c for c in customerIds if not 0 <= c < self.model.numUser]
        if bad:
            raise ValueError(f"unknown customer ids {bad[:5]}")
        if not customerIds or not self.productIds:
            return [{} for _ in customerIds]
        dev = self.model.device
        items = torch.as_tensor(np.asarray(self.productIds, dtype=np.int32)).to(dev)
        I = items.numel()
        k = min(int(numberOfItem), I)
        if not 1 <= k <= 32:
            raise ValueError("numberOfItem must be between 1 and 32 (the device top-k keeps at most 32 per row)")
        out = []
        per = max(1, (1 << 22) // I)                                      # <= 4 M (customer, product) pairs per pass
        for a in range(0, len(customerIds), per):
            chunk = customerIds[a:a + per]
            u = torch.as_tensor(np.asarray(chunk, dtype=np.int32)).to(dev).repeat_interleave(I)
            pred, _ = self.model.predict_on_batch(u, items.repeat(len(chunk)))
            scores = pred.view(len(chunk), I)
            scores = torch.where(scores < 1.0, scores, torch.full_like(scores, float("-inf")))   # filter(... < 1.0), :46
            v, ix = H.topk_rows(scores.contiguous(), k)
            v, ix = v.cpu().numpy(), ix.cpu().numpy()
            for r in range(len(chunk)):
                out.append({self.productIds[j]: '%.9f' % s for s, j in zip(v[r], ix[r]) if np.isfinite(s)})
        return out

    def predictForUser(self, customerId, numberOfItem=5):
        return self.predictForUsers([customerId], numberOfItem)[0]

    # This model only supports predict (NCFModel.py:53-55)
    def readyToTrain(self):
        return False

    def getPredictableUsers(self):
        return self.customerIds

    def loadTrainData(self):
        """customer_id,normalized_customer_id,material,product_id,rating_type (NCFModel.py:60-64): the distinct product
        ids and normalized customer ids of the file, in order of first appearance (`.unique()`)."""
        from .interactions import read_csv_columns
        with self.dataStore.openFile(self.trainData) as f:
            cols = read_csv_columns(f, "ncf")
        first = lambda a: list(dict.fromkeys(np.asarray(a).tolist()))
        self.productIds = first(cols["item"])
        self.customerIds = first(cols["user"])


def fit_nfc_plain(train, test, epochs=20, batch_size=50000, lr=0.005, dropout=0.2, seed=42, shuffle_seed=7, device=None,
                  tensor_cores=False, verbose=0):
    """The training script trainers/NFC_plain.py as a function: `train` / `test` are (customer, product, rating_type)
    column triples (its two CSVs, columns normalized_customer_id / product_id / rating_type, :72-73).
      tables   : num_customers + 1 rows with num_customers = #distinct customers over both files, num_materials + 1
                 rows with num_materials = the largest product id (:79-82, :116-126);
      model    : latent 10, Dense 100 / 50 / 10 sigmoid with BatchNorm after fc-1 / fc-2, dropout 0.2, head
                 [pred_mf, pred_mlp], BCE, Adam(0.005) (:109-155);
      fit      : explicit labels from the file (no negative sampling), batch 50 000, 20 epochs, rows reshuffled every
                 epoch (`shuffle(train)` :85 and fit(shuffle=True) :165 -- seeded here);
      after it : predictions on the test file rounded to 2 decimals -> mean absolute error (:178-180), evaluate (:183).
    Returns {'model', 'history': [epoch losses], 'test_mae_rounded', 'evaluate': [loss, mse, mae, binary_accuracy]}."""
    from . import pipeline as PL
    dev = torch.device(device) if device is not None else torch.device(f"cuda:{torch.cuda.current_device()}")
    tu, ti, ty = (np.asarray(c) for c in train)
    su, si, sy = (np.asarray(c) for c in test)
    num_customers = len(np.unique(np.concatenate([tu, su])))
    num_materials = int(max(ti.max(initial=0), si.max(initial=0)))
    if max(tu.max(initial=0), su.max(initial=0)) > num_customers:
        raise ValueError("normalized customer ids must lie in [0, number of distinct customers] (Embedding(num_customers + 1))")
    net = NeuMFNet(num_customers + 1, num_materials + 1, 10, hidden=(100, 50, 10), act="sigmoid", loss="bce", learning_rate=lr,
                   dropout=dropout, seed=seed, head_order="mf_h3", device=dev, tensor_cores=tensor_cores)
    u = torch.from_numpy(np.ascontiguousarray(tu, dtype=np.int32)).to(dev)
    i = torch.from_numpy(np.ascontiguousarray(ti, dtype=np.int32)).to(dev)
    y = torch.from_numpy(np.ascontiguousarray(ty, dtype=np.float32)).to(dev)
    n = u.numel()
    nb = (n + batch_size - 1) // batch_size
    history = []
    for e in range(epochs):
        perm = PL.epoch_permutation(n, shuffle_seed, e, device=dev)          # rows reshuffled per epoch, on the device
        ue, ie, ye = u[perm].contiguous(), i[perm].contiguous(), y[perm].contiguous()
        losses = net.train_steps(ue, ie, ye, batch_size, np.arange(nb), epoch=e)
        history.append(float(losses.double().mean().item()))
        if verbose:
            print(f"Epoch {e + 1}/{epochs} - loss: {history[-1]:.4f}")
    tu_d = torch.from_numpy(np.ascontiguousarray(su, dtype=np.int32)).to(dev)
    ti_d = torch.from_numpy(np.ascontiguousarray(si, dtype=np.int32)).to(dev)
    ty_d = torch.from_numpy(np.ascontiguousarray(sy, dtype=np.float32)).to(dev)
    pred, loss = net.predict_on_batch(tu_d, ti_d, ty_d)
    y_hat = torch.round(pred * 100.0) / 100.0                               # np.round(..., decimals=2), :178
    err = pred - ty_d
    return {"model": net, "history": history,
            "test_mae_rounded": float((y_hat - ty_d).abs().mean().item()),
            "evaluate": [float(loss.item()), float((err * err).mean().item()), float(err.abs().mean().item()),
                         float(((pred > 0.5).float() == ty_d).float().mean().item())]}
