"""Metrics surface of the training loop (SURVEY §8f item 3): the reference's ``Logger`` (JSONL +
summary), ``TensorBoardLogger`` and ``MetricsTracker`` interfaces (src/utils/logger.py:28-302),
so dashboards and scripts that read the reference's logs read ours: one JSON object per line with
``step``/``time``/``timestamp`` plus the metrics, ``<name>_summary.json`` with mean/std/min/max/last
per metric, and the TensorBoard tags of scripts/train.py:247-258 (``performance/*``, ``training/*``), plus
``evaluation/*`` for the held-out evaluations of ``b200.eval_interval``.

The values are produced by on-device episode reductions (train.py), not by a per-episode Python
loop; only the writer side lives here.
"""
import collections
import datetime
import json
import math
import os
import time

import numpy as np


def _plain(x):
    """numpy / torch scalars and arrays -> JSON-serialisable Python objects."""
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, np.ndarray):
        return x.tolist()
    if isinstance(x, np.generic):
        return x.item()
    if hasattr(x, "detach") and hasattr(x, "cpu"):          # torch tensor
        x = x.detach().cpu()
        return x.item() if x.numel() == 1 else x.tolist()
    return x


def _is_number(x):
    return isinstance(x, (int, float, np.integer, np.floating)) and not isinstance(x, bool)


class Logger:
    """JSON-lines metric log (reference src/utils/logger.py:28-131)."""

    def __init__(self, log_dir, name="training"):
        os.makedirs(log_dir, exist_ok=True)
        self.log_dir, self.name = str(log_dir), name
        self.start_time = time.time()
        stamp = datetime.datetime.now().strftime("%Y%m%d_%H%M%S")
        self.log_file = os.path.join(self.log_dir, "%s_%s.jsonl" % (name, stamp))
        self.metrics_history = collections.defaultdict(list)
        self.step = 0

    def log(self, metrics, step=None):
        self.step = int(step) if step is not None else self.step + 1
        metrics = _plain(metrics)
        # the caller's own 'step' key (scripts/train.py:236) wins over ours, as in the reference
        record = {"step": self.step, "time": time.time() - self.start_time,
                  "timestamp": datetime.datetime.now().isoformat(), **metrics}
        for k, v in metrics.items():
            if _is_number(v):
                self.metrics_history[k].append(float(v))
        with open(self.log_file, "a") as f:
            f.write(json.dumps(record) + "\n")
        return record

    def get_recent(self, metric, n=100):
        return self.metrics_history[metric][-n:]

    def get_mean(self, metric, n=100):
        vals = self.get_recent(metric, n)
        return float(np.mean(vals)) if vals else 0.0

    def print_metrics(self, metrics):
        sec = int(time.time() - self.start_time)
        print("\n[Step {:,}] [{:02d}:{:02d}:{:02d}]".format(self.step, sec // 3600, sec % 3600 // 60, sec % 60))
        for k, v in metrics.items():
            print("  %s: %s" % (k, "%.4f" % v if isinstance(v, float) else v))

    def save_summary(self):
        out = {"name": self.name, "total_steps": self.step, "total_time": time.time() - self.start_time, "metrics": {}}
        for k, vals in self.metrics_history.items():
            a = np.asarray(vals, np.float64)
            out["metrics"][k] = {"mean": float(a.mean()), "std": float(a.std()), "min": float(a.min()),
                                 "max": float(a.max()), "last": float(a[-1])}
        path = os.path.join(self.log_dir, "%s_summary.json" % self.name)
        with open(path, "w") as f:
            json.dump(out, f, indent=2)
        return path


class TensorBoardLogger:
    """Thin SummaryWriter front end (reference logger.py:134-218); a no-op when tensorboard is
    not installed."""

    def __init__(self, log_dir, name="training"):
        self.step = 0
        try:
            from torch.utils.tensorboard import SummaryWriter
            self.writer = SummaryWriter(log_dir=os.path.join(str(log_dir), name))
            self.enabled = True
        except Exception:                                    # ImportError or a broken TB install
            self.writer, self.enabled = None, False

    def _at(self, step):
        if step is not None:
            self.step = int(step)
        return self.step

    def log_scalar(self, tag, value, step=None):
        s = self._at(step)
        if self.enabled:
            self.writer.add_scalar(tag, float(_plain(value)), s)

    def log_scalars(self, main_tag, values, step=None):
        s = self._at(step)
        if self.enabled:
            self.writer.add_scalars(main_tag, {k: float(_plain(v)) for k, v in values.items()}, s)

    def log_histogram(self, tag, values, step=None):
        s = self._at(step)
        if self.enabled:
            self.writer.add_histogram(tag, np.asarray(_plain(values)), s)

    def log_image(self, tag, image, step=None):
        s = self._at(step)
        if self.enabled:
            self.writer.add_image(tag, image, s, dataformats="HWC")

    def log_text(self, tag, text, step=None):
        s = self._at(step)
        if self.enabled:
            self.writer.add_text(tag, text, s)

    def log_metrics(self, metrics, step=None):
        s = self._at(step)
        for k, v in metrics.items():
            self.log_scalar(k, v, s)

    def close(self):
        if self.enabled:
            self.writer.close()


class MetricsTracker:
    """Rolling-window statistics (reference logger.py:221-287)."""

    def __init__(self, window_size=100):
        self.window_size = window_size
        self.metrics = collections.defaultdict(lambda: collections.deque(maxlen=self.window_size))

    def add(self, name, value):
        self.metrics[name].append(float(_plain(value)))

    def add_many(self, name, values):
        """Append a batch (e.g. the scores of all episodes that finished in one vec step)."""
        self.metrics[name].extend(float(v) for v in np.asarray(_plain(values)).ravel())

    def _vals(self, name):
        return np.asarray(self.metrics[name], np.float64) if name in self.metrics else np.empty(0)

    def get_mean(self, name):
        v = self._vals(name)
        return float(v.mean()) if v.size else 0.0

    def get_std(self, name):
        v = self._vals(name)
        return float(v.std()) if v.size else 0.0

    def get_min(self, name):
        v = self._vals(name)
        return float(v.min()) if v.size else 0.0

    def get_max(self, name):
        v = self._vals(name)
        return float(v.max()) if v.size else 0.0

    def get_last(self, name):
        v = self._vals(name)
        return float(v[-1]) if v.size else 0.0

    def get_summary(self, name):
        return {"mean": self.get_mean(name), "std": self.get_std(name), "min": self.get_min(name),
                "max": self.get_max(name), "last": self.get_last(name)}

    def get_all_summaries(self):
        return {k: self.get_summary(k) for k in self.metrics}

    def reset(self):
        self.metrics.clear()


EVAL_KEYS = ("eval_mean_score", "eval_std_score", "eval_max_score", "eval_min_score", "eval_mean_length",
             "eval_finished", "eval_wall_s")


# TensorBoard tags of scripts/train.py:247-258, from one JSONL row of train.py; evaluation/* for held-out evaluations
def tensorboard_tags(row):
    tags = {"performance/avg_score": row["avg_score"], "performance/max_score": row["max_score"],
            "performance/best_score": row["best_score"], "performance/avg_length": row["avg_length"],
            "performance/fps": row["fps"]}
    for k in ("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction"):
        if k in row and not (isinstance(row[k], float) and math.isnan(row[k])):
            tags["training/" + k] = row[k]
    for k in EVAL_KEYS:                       # rows of updates with a held-out evaluation (train.py)
        if k in row:
            tags["evaluation/" + k[len("eval_"):]] = row[k]
    return tags
