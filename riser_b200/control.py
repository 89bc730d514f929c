"""The ReadUntil loop with a batched body: a drop-in for ``SequencerControl`` of riser/control.py.

What the sequencer, the log and the CSV see is what riser/control.py:4-153 produces -- the take-over and
stop warnings, one CSV row per assessed read in read order, ``unblock`` for rejects, ``stop_receiving`` for
every read that needs no further look, the per-minute tally, the poly(A)-cache wipe at 1000 entries.  How a
poll is worked through is different: the reference walks the reads of a poll one by one through trim ->
gate -> normalise -> classify -> decide (control.py:31-93); here the whole poll goes to
``BatchedClassifier.classify_batch`` once, the decision codes come back as one array, and the rows and the
three read lists are cut out of that array.
"""
import collections
import time

import numpy as np

from .pipeline import BatchedClassifier, DECISION_NAMES, SKIPPED, ACCEPT, REJECT, NO_DECISION
from .preprocess import signal_dtype

CSV_HEADER = 'batch_start,read_id,channel,sig_length,models,prob_targets,threshold,mode,decision\n'   # control.py:146
TAKE_OVER_NOTICE = ('The sequencing run is being controlled by RISER, reads that are '
                    'not in the target class will be ejected from the pore.')                         # control.py:13-14
PROGRESS_PERIOD_S = 60                                                                                # control.py:19,116
LATENCY_HISTORY = 4096       # polls whose latency / size SequencerControl remembers


class _MinuteTally:
    """assessed / accepted / rejected since the last progress line (control.py:21-23,108-117)."""
    def __init__(self, logger, now):
        self.logger = logger
        self.due = now + PROGRESS_PERIOD_S
        self.assessed = self.accepted = self.rejected = 0

    def add(self, assessed, accepted, rejected):
        self.assessed += assessed
        self.accepted += accepted
        self.rejected += rejected

    def maybe_report(self, batch_start):
        if batch_start <= self.due:
            return
        self.logger.info(f"In the last minute {self.assessed} signals "
                         f"were assessed, {self.accepted} were "
                         f"accepted and {self.rejected} were rejected")
        self.assessed = self.accepted = self.rejected = 0
        self.due = batch_start + PROGRESS_PERIOD_S


def _sequencer_key(read):
    """What unblock / stop_receiving want for a read: its number with minknow-api <= v5, its id from v6 on
    (control.py:137-143)."""
    return read.number if hasattr(read, "number") else read.id


class SequencerControl():
    def __init__(self, client, models, processor, logger, out_file, warm_up_batches=()):
        """Arguments as riser/control.py:5.  ``warm_up_batches`` (additive, optional): batch sizes whose launch
        plans and CUDA graphs are built at the start of ``target`` instead of during the first polls that see
        them (e.g. ``(512,)`` for a MinION)."""
        self.client = client
        self.models = models
        self.proc = processor
        self.logger = logger
        self.out_filename = out_file
        self.classifier = BatchedClassifier(models, processor)
        self.classifier_f32 = None     # built on the first poll of calibrated (float32) signal
        self.warm_up_batches = tuple(warm_up_batches)
        # Instrumentation (additive): seconds from "batch in hand" to "decisions on host" and the batch size of
        # the most recent non-empty polls.  Bounded -- ReadUntil's get_read_chunks does not block, so an idle
        # client is polled tens of thousands of times a second and a run lasts days.
        self.batch_latencies = collections.deque(maxlen=LATENCY_HISTORY)
        self.batch_sizes = collections.deque(maxlen=LATENCY_HISTORY)

    # ------------------------------------------------------------------ riser.py's three calls
    def start(self):
        self.client.start_streaming_reads()
        self.logger.info('Live read stream started.')

    def finish(self):
        self.client.reset()
        self.logger.info('Client reset and live read stream ended.')

    def target(self, mode, duration_h, threshold, unblock_duration=0.1):
        self.client.send_warning(TAKE_OVER_NOTICE)
        if self.warm_up_batches:
            calibrated = np.dtype(getattr(self.client, "signal_dtype", np.int16)) == np.float32
            clf = self._classifier_f32() if calibrated else self.classifier
            clf.warm_up(self.warm_up_batches, threshold, mode)
        model_names = ";".join(m.target for m in self.models)
        polyA_cache = {}       # one dict for the run; classify_batch stores found ends and wipes it at 1000 entries
        with open(f'{self.out_filename}.csv', 'a') as sink:
            sink.write(CSV_HEADER)
            began = time.monotonic()
            deadline = began + duration_h * 3600
            tally = _MinuteTally(self.logger, began)
            while self.client.is_running() and time.monotonic() < deadline:
                self._poll(sink, tally, polyA_cache, model_names, mode, threshold, unblock_duration)
            self.client.send_warning('RISER has stopped running.')
            if not self.client.is_running():
                self.logger.info('Client has stopped.')
            if time.monotonic() > deadline:
                self.logger.info(f'RISER has timed out after {duration_h} '
                                 'hours as requested.')

    def _classifier_f32(self):
        if self.classifier_f32 is None:
            self.classifier_f32 = BatchedClassifier(self.models, self.proc, signal_dtype=np.float32)
        return self.classifier_f32

    def _classifier_for(self, signals):
        """The classifier for a poll's arrays: the float32 one when they are float32 (a client run with calibrated
        signal), the int16 one otherwise; a poll that mixes float32 with other dtypes raises TypeError."""
        return self._classifier_f32() if signal_dtype(signals) == np.float32 else self.classifier

    # ------------------------------------------------------------------ one poll
    def _poll(self, sink, tally, polyA_cache, model_names, mode, threshold, unblock_duration):
        batch_start = time.monotonic()
        batch = list(self.client.get_read_batch())
        if not batch:
            # nothing arrived: the reference's loop body does not run and its two client calls get empty lists
            # (control.py:100-106); no device work, nothing recorded
            self.client.reject_reads([], unblock_duration)
            self.client.finish_processing_reads([])
            tally.maybe_report(batch_start)
            return
        signals = [self.client.get_raw_signal(read) for _, read in batch]
        t0 = time.monotonic()
        clf = self._classifier_for(signals)
        res = clf.classify_batch(signals, [read.id for _, read in batch], polyA_cache, threshold, mode)
        self.batch_latencies.append(time.monotonic() - t0)
        self.batch_sizes.append(len(batch))

        codes = np.asarray(res.decisions)
        assessed = np.flatnonzero(codes != SKIPPED)          # the others hit a `continue` (control.py:50,56)
        stamp = f'{batch_start:.0f}'
        sink.writelines(
            f'{stamp},{batch[i][1].id},{batch[i][0]},{int(res.sig_len[i])},{model_names},'
            f'{";".join(str(float(p)) for p in res.p_on[i])},{threshold},{mode},{DECISION_NAMES[int(codes[i])]}\n'
            for i in assessed)

        def keyed(code):
            return [(batch[i][0], _sequencer_key(batch[i][1])) for i in np.flatnonzero(codes == code)]

        rejects, accepts, undecided = keyed(REJECT), keyed(ACCEPT), keyed(NO_DECISION)
        self.client.reject_reads(rejects, unblock_duration)
        # rejected, accepted and exhausted (max length, still undecided) reads need no further look
        self.client.finish_processing_reads(rejects + accepts + undecided)
        tally.add(len(assessed), len(accepts), len(rejects))
        tally.maybe_report(batch_start)
