"""``DATALOADERS`` / ``dataloader_factory`` of NN/dataloaders/__init__.py:11-14,69-89 over the device-side producers.

Same contract: ``dataloader_factory(args) -> (train, val, test)`` loaders whose batches have the reference's wire format
(SURVEY.md 8a19) -- built on the GPU: histories live there as a CSR, a training batch is one kernel launch
(``rbm_bert_cloze_batch`` / ``rbm_sas_train_batch``), evaluation negatives are drawn by ``rbm_negative_samples`` and evaluation
batches assembled by ``rbm_eval_batch``.  Differences, on purpose: no pickle caches are written (``Data/Processed/*.p``,
negative-sample ``*.pkl``), worker processes are not needed (``worker_number`` is ignored), and the unused training negatives
of ``AbstractDataloader.__init__`` (NN/dataloaders/base.py:26-31: generated, never read by either loader) are not generated.
"""
import os
import pickle
from abc import ABCMeta, abstractmethod

from .device import DeviceBertTrainLoader, DeviceSasTrainLoader, DeviceNegativeSampler, DeviceEvalLoader
from .partition import data_partition


class AbstractDataloader(metaclass=ABCMeta):
    """NN/dataloaders/base.py:12-45: dataset = [user_train, user_valid, user_test, usernum, itemnum]."""

    def __init__(self, args, dataset):
        self.args = args
        self.train, self.val, self.test = dataset[0], dataset[1], dataset[2]
        self.user_count, self.item_count = dataset[3], dataset[4]
        args.num_items = self.item_count  # NN/dataloaders/base.py:22
        self.max_len = args.max_len
        self.device = args.device
        self.seed = int(getattr(args, "dataloader_random_seed", 0) or 0)
        # full-catalogue evaluation ranks every item the user has not seen: no sampled negatives
        self.full_catalogue = bool(getattr(args, "full_catalogue_eval", False))
        self.test_negative_samples = None if self.full_catalogue else DeviceNegativeSampler(
            self.train, self.val, self.test, self.user_count, self.item_count, args.test_negative_sample_size,
            args.test_negative_sampling_seed, self.device, code=args.test_negative_sampler_code).get_negative_samples()

    @classmethod
    @abstractmethod
    def code(cls):
        pass

    @abstractmethod
    def _train_loader(self):
        pass

    mask_token = -1

    def _eval_loader(self, mode):
        """NN/dataloaders/bert.py:44-62, sas.py:49-62: validation scores train histories against the validation item, the test
        split appends the validation item to the history first.  ``args.full_catalogue_eval``: batches of (seq, answers,
        exclude) for ranking the whole catalogue minus that history (see ``DeviceEvalLoader``)."""
        if mode == "val":
            history, answers, bs = self.train, self.val, self.args.val_batch_size
        else:
            history = [list(seq) + [self.val[u][0]] for u, seq in enumerate(self.train)]
            answers, bs = self.test, self.args.test_batch_size
        return DeviceEvalLoader(history, answers, self.test_negative_samples, self.max_len, bs, self.device, mask_token=self.mask_token,
                                full_catalogue=self.full_catalogue)

    def get_pytorch_dataloaders(self):
        return self._train_loader(), self._eval_loader("val"), self._eval_loader("test")


class BertDataloader(AbstractDataloader):
    """NN/dataloaders/bert.py:8-62."""

    def __init__(self, args, dataset):
        super().__init__(args, dataset)
        self.mask_prob = args.bert_mask_prob
        self.CLOZE_MASK_TOKEN = self.item_count + 1
        self.mask_token = self.CLOZE_MASK_TOKEN

    @classmethod
    def code(cls):
        return 'bert'

    def _train_loader(self):
        return DeviceBertTrainLoader(self.train, self.max_len, self.mask_prob, self.item_count, self.args.train_batch_size, self.device,
                                     seed=self.seed)


class SASDataLoader(AbstractDataloader):
    """NN/dataloaders/sas.py:11-62."""

    @classmethod
    def code(cls):
        return 'sas'

    def _train_loader(self):
        return DeviceSasTrainLoader(self.train, self.max_len, self.item_count, self.args.train_batch_size, self.device, seed=self.seed)


DATALOADERS = {BertDataloader.code(): BertDataloader, SASDataLoader.code(): SASDataLoader}


def dataloader_factory(args, dataset=None):
    """NN/dataloaders/__init__.py:69-89.  ``dataset`` may be passed directly; else ``args.processed_dataset_path`` (pickle) when
    ``args.load_processed_dataset``, else the text file ``args.data_path`` (or ``<args.data_root or 'Data'>/<args.data_name>``)."""
    if dataset is None:
        if getattr(args, "load_processed_dataset", False):
            with open(os.path.normpath(args.processed_dataset_path), "rb") as fh:
                dataset = pickle.load(fh)
        else:
            path = getattr(args, "data_path", None) or os.path.join(getattr(args, "data_root", None) or "Data", args.data_name)
            dataset = data_partition(path, args.max_len, args.prop_sliding_window)
    if args.model_code not in DATALOADERS:
        raise KeyError("unknown model_code %r (have %s)" % (args.model_code, sorted(DATALOADERS)))
    loader = DATALOADERS[args.model_code](args, dataset)
    return loader.get_pytorch_dataloaders()
