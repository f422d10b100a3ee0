"""Host-buffer serving loop for the encoder: the public end-to-end entry point.

``EncoderPipeline.run`` takes batches that live in (pinned) HOST memory and returns encoder outputs in
HOST memory.  All arithmetic happens in the sm_100a kernels; PyTorch only moves bytes and orders
streams:

  * one copy-in stream (pinned host batch -> device), one copy-out stream (result -> pinned host);
  * ``lanes`` compute streams.  Batch i runs on lane ``i % lanes`` (fbank CMVN + encoder forward; each
    lane replays its own CUDA graph, so it owns its activations).  Every kernel of the forward is a
    persistent grid of one CTA (pair) per SM whose last wave leaves SMs idle; with two batches in
    flight the CTAs of one lane's kernel start on the SMs the other lane's kernel has already left
    (measured at cfg2: 2.70 -> 2.58 ms/step, profiles/r01g_overlap_probe.txt);
  * the forward is used through its asynchronous half (``encoder.launch``): the host never waits for
    batch i before batch i+1 .. i+lanes are enqueued, so the only host synchronisation of the forward
    (the new lengths after CTC compression, needed for the output SHAPE) is hidden behind queued work.

The per-batch work is exactly ``apply_mv_norm`` (data/fbank_dataset.py:44-45) followed by
``ConvolutionalTransformerEncoder.forward`` (models/conv_transformer.py:195-276).
"""
import collections

import torch

from . import ops


class EncoderPipeline:
    def __init__(self, encoder, normalize=True, device=None, lanes=None):
        if lanes is None:  # two lanes measured best (profiles/r01g_overlap_probe.txt, r02y)
            lanes = 2
        self.enc = encoder
        self.normalize = normalize
        self.device = device or next(encoder.parameters()).device
        # eager launches share lazily created tables across lanes: keep one lane unless graphs are on
        self.lanes = min(4, max(1, int(lanes))) if encoder.use_cuda_graph else 1
        self.s_in = torch.cuda.Stream(self.device)
        self.s_lane = [torch.cuda.Stream(self.device) for _ in range(self.lanes)]
        self.s_out = torch.cuda.Stream(self.device)
        self._dev_in = {}    # (slot, shape) -> device staging buffer
        self._host_out = {}  # (slot, shape, dtype) -> pinned host buffer
        self._n_in = self.lanes + 2
        self._consumed = [None] * self._n_in  # event: CMVN / encoder finished reading input slot
        with torch.cuda.device(self.device):
            encoder._prepared_active()  # derive the operand formats once, before any lane uses them
            torch.cuda.synchronize(self.device)

    def _in_buffer(self, slot, shape):
        key = (slot, tuple(shape))
        if key not in self._dev_in:
            self._dev_in[key] = torch.empty(shape, dtype=torch.float32, device=self.device)
        return self._dev_in[key]

    def _out_buffer(self, slot, shape, dtype):
        key = (slot, tuple(shape), dtype)
        if key not in self._host_out:
            self._host_out[key] = torch.empty(shape, dtype=dtype).pin_memory()
        return self._host_out[key]

    def _enqueue(self, i, batch):
        """H2D of batch i on the copy-in stream, then CMVN + the asynchronous half of the forward on
        lane i % lanes.  Nothing here waits on the host."""
        x_host, lengths = batch
        slot = i % self._n_in
        if x_host.is_cuda:  # device-resident batch (run_device): nothing to stage
            buf, ev_in = x_host, None
        else:
            buf = self._in_buffer(slot, x_host.shape)
            with torch.cuda.stream(self.s_in):
                if self._consumed[slot] is not None:
                    self.s_in.wait_event(self._consumed[slot])
                buf.copy_(x_host, non_blocking=True)
                ev_in = torch.cuda.Event()
                ev_in.record(self.s_in)
        lane = i % self.lanes
        s = self.s_lane[lane]
        with torch.cuda.stream(s):
            if ev_in is not None:
                s.wait_event(ev_in)
            self.enc.graph_lane = lane
            try:
                if self.normalize:
                    len32 = lengths.to(torch.int32).to(self.device, non_blocking=True)
                    # CMVN writes straight into the lane's graph input when that graph already exists
                    x = ops.cmvn(buf, len32, out=self.enc.static_input(*buf.shape, buf.device))
                else:
                    x = buf
                handle = self.enc.launch(x, lengths)
            finally:
                self.enc.graph_lane = 0
            ev_done = torch.cuda.Event()
            ev_done.record(s)
        self._consumed[slot] = ev_done
        return handle, ev_done

    def _collect(self, j, handle, ev_done, to_host=True):
        """Blocking half for batch j: exact output shape (waits for the batch's new lengths; the batches
        queued behind it keep the GPU busy).  Host mode: the D2H copy is enqueued on the copy-out
        stream and returned as (event, host tensor, host lengths) -- the caller waits for it AFTER it
        has enqueued the next batch."""
        if not to_host:
            # hand the result over to the caller's stream (ordered after batch j, not after the
            # batches queued behind it on the lane)
            self._caller.wait_event(ev_done)
            with torch.cuda.stream(self._caller):
                out = self.enc.finish(handle)
            for t in (out.encoder_out, out.encoder_padding_mask, getattr(out, "ctc_padding_mask", None)):
                if t is not None:
                    t.record_stream(self._caller)  # allocated on the lane's stream
            return out
        with torch.cuda.stream(self.s_out):
            out = self.enc.finish(handle)
            self.s_out.wait_event(ev_done)
            eo = out.encoder_out
            host = self._out_buffer(j & 1, eo.shape, eo.dtype)
            host.copy_(eo, non_blocking=True)
            ev_out = torch.cuda.Event()
            ev_out.record(self.s_out)
        hl = torch.tensor(handle["out_len_host"], dtype=handle["len_dtype"])  # set by finish (host)
        return ev_out, host, hl, out  # `out` keeps the device tensor alive until the copy has finished

    def run(self, batches):
        """``batches``: iterable of ``(src_tokens [B,T,F] fp32 host tensor, src_lengths [B] int64 host
        tensor)``.  Yields ``(encoder_out [T'',B,D] fp32 host tensor, out_lengths [B] host tensor)`` in
        order.  A yielded ``encoder_out`` is a view of a reusable pinned buffer: consume it before
        asking for the batch after next."""
        return self._run(batches, True)

    def run_device(self, batches):
        """Same loop for batches that already live on the device: yields the encoder's output tuples
        (device tensors, usable on the caller's current stream).  ``ctc_out`` aliases a buffer of the lane's CUDA
        graph: it is valid until ``lanes`` more batches of the same shape have been yielded."""
        return self._run(batches, False)

    def _run(self, batches, to_host):
        caller = self._caller = torch.cuda.current_stream(self.device)
        for s in self.s_lane:
            s.wait_stream(caller)
        inflight = collections.deque()
        copying = None  # host mode: the batch whose D2H copy is in flight

        def deliver(c):
            c[0].synchronize()
            return c[1], c[2]

        for i, batch in enumerate(batches):
            inflight.append((i,) + self._enqueue(i, batch))
            if copying is not None:  # its copy has been running while batch i was enqueued
                yield deliver(copying)
                copying = None
            if len(inflight) > self.lanes:  # batches i-lanes+1 .. i stay queued behind this wait
                j, handle, ev_done = inflight.popleft()
                r = self._collect(j, handle, ev_done, to_host)
                if to_host:
                    copying = r
                else:
                    yield r
        while inflight or copying is not None:
            if copying is not None:
                yield deliver(copying)
                copying = None
            if inflight:
                j, handle, ev_done = inflight.popleft()
                r = self._collect(j, handle, ev_done, to_host)
                if to_host:
                    copying = r
                else:
                    yield r
        for s in self.s_lane:
            caller.wait_stream(s)
