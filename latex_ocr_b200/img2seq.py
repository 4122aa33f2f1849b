"""Img2SeqModel — the trainer surface of model/img2seq_torch.py:64-172 + model/base_torch.py:45-206
(build_train / getLoss / _run_train_epoch / train) on the B200-native encoder and decoder.

``getLoss`` keeps the reference semantics exactly (img2seq_torch.py:136-172): every row's caption
length is the padded length (:144), targets are captions[:, 1:] (:147), loss = CE(mean over packed
positions, PADs included) + 1.0 * mean((1 - sum_t alpha)^2) (:151-159), backward, Adam step on the
decoder then the encoder (:162-170), returns ``-loss`` (:172).  The ``lr`` and ``dropout`` arguments
are ignored exactly like the reference ignores them (SURVEY.md quirk Q3).
"""
import ctypes
import os
import time

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr
from .decoder import DecoderWithAttention
from .encoder import EncoderCNN
from .params import LRUCache


class Img2SeqModel:
    def __init__(self, config, dir_output=None, vocab=None, device=None, precision=None, impl=None, n_tok=None):
        self._config = config
        self._dir_output = dir_output
        self._vocab = vocab
        dev = device or getattr(config, "device", "cuda")
        if not str(dev).startswith("cuda"):
            raise _lib.LatexOcrB200Error("latex_ocr_b200 runs on CUDA devices only (device=%r)" % (dev,))
        self.device = torch.device(dev)
        self.precision = precision or getattr(config, "precision", "bf16")
        # kernels: "tc" = tcgen05/TMA convolutions and GEMMs (bf16 storage only), "simt" = CUDA-core twins (fp32 tight-parity mode)
        self.impl = impl or getattr(config, "impl", "tc" if self.precision == "bf16" else "simt")
        self._n_tok = n_tok if n_tok is not None else (vocab.n_tok if vocab is not None else None)
        self.encoder = None
        self.decoder = None
        self.use_graph = bool(getattr(config, "cuda_graph", False))
        self._graphs = LRUCache()  # captured train-step graphs, one per (shapes, mode): bounded like the workspaces
        self.dist = None          # set by latex_ocr_b200.dist.attach(model)
        self.lr = float(getattr(config, "lr_init", 1e-3))

    # --- model/base_torch.py:45-71 -------------------------------------------------------------
    def build_train(self, config=None):
        config = config or self._config
        self.getModel("Img2Seq")
        self.getOptimizer(getattr(config, "lr_method", "adam"), float(getattr(config, "lr_init", 1e-3)))
        return self

    def build_pred(self, config=None):
        self.getModel("Img2Seq")
        return self

    def getModel(self, model_name="Img2Seq"):
        """img2seq_torch.py:69-83 (only the Img2Seq branch is on the hot path)."""
        if model_name != "Img2Seq":
            raise NotImplementedError("model_name=%r: only 'Img2Seq' is implemented" % model_name)
        self.encoder = EncoderCNN(self._config, device=self.device, precision=self.precision, impl=self.impl)
        self.decoder = DecoderWithAttention(attention_dim=512, embed_dim=512, decoder_dim=512, vocab_size=self._n_tok,
                                            dropout=0.5, device=self.device, precision=self.precision, impl=self.impl)
        return self

    def getOptimizer(self, lr_method="adam", lr=0.001):
        """img2seq_torch.py:85-88: two Adam optimisers with torch defaults (one fused launch each)."""
        if str(lr_method).lower() != "adam":
            raise NotImplementedError("lr_method=%r: the torch path of the reference always builds Adam" % lr_method)
        self.lr = float(lr)
        self.encoder.store.ensure_adam(lr)
        self.decoder.store.ensure_adam(lr)

    def set_lr(self, lr):
        """Learning rate of both fused Adam optimisers (a device scalar read by the kernel: works under graph replay)."""
        self.lr = float(lr)
        self.encoder.store.set_lr(lr)
        self.decoder.store.set_lr(lr)

    def train_mode(self, flag=True):
        self.encoder.train(flag)
        self.decoder.train(flag)

    # --- the fused train step --------------------------------------------------------------------
    @staticmethod
    def _trainable_ranges(store, module):
        """Contiguous {offset, count} ranges of the flat store owned by parameters with requires_grad=True, or None when
        nothing is frozen."""
        frozen = {p_._lo_store_name for p_ in module.parameters() if not p_.requires_grad}
        if not frozen:
            return None
        ranges = []
        for name, (off, n, _) in sorted(store.offsets.items(), key=lambda kv: kv[1][0]):
            if name in frozen:
                continue
            if ranges and ranges[-1][0] + ranges[-1][1] == off:
                ranges[-1][1] += n
            else:
                ranges.append([off, n])
        return ranges

    def _adam(self, store, grad_scale=1.0, module=None):
        L = _lib.lib()
        ranges = self._trainable_ranges(store, module) if module is not None else None
        if ranges is None:
            check(L.lo_adam_step(ptr(store.master), ptr(store.grad), ptr(store.m), ptr(store.v), ptr(store.shadow), store.numel,
                                 ptr(store.adam_state), 0.9, 0.999, 1e-8, float(grad_scale), stream_ptr()))
            return
        # fine_tune()/fine_tune_embeddings() (seq2seq_torch.py:102-113, :246-253): torch.optim.Adam skips parameters without a
        # gradient, so frozen slices see neither moment decay nor an update
        import ctypes
        flat = [x for r in ranges for x in r]
        arr = (ctypes.c_int64 * max(len(flat), 1))(*flat)
        check(L.lo_adam_step_ranges(ptr(store.master), ptr(store.grad), ptr(store.m), ptr(store.v), ptr(store.shadow), arr, len(ranges),
                                    ptr(store.adam_state), 0.9, 0.999, 1e-8, float(grad_scale), stream_ptr()))

    def _step_body(self, img, caps, decode_lengths, dropout_mask):
        """encoder fwd -> decoder fwd + loss -> decoder bwd -> encoder bwd -> (grad all-reduce) -> Adam x2.
        img: CUDA fp32 [N,1,H,W]; caps: CUDA int64 [N,L] sorted rows.  Returns the device loss vector."""
        N = img.shape[0]
        enc_out = self.encoder.forward_raw(img, need_grad=True)
        R = enc_out.shape[1] * enc_out.shape[2]
        enc_flat = enc_out.view(N, R, enc_out.shape[3])
        ws = self.decoder.run_forward(enc_flat, caps, decode_lengths, with_loss=True, need_grad=True, dropout_mask=dropout_mask)
        self.decoder.run_backward(ws)
        scale = 1.0
        if self.dist is not None:
            self.dist.reduce_async(self.decoder.store.grad)        # decoder bucket flies while the encoder backward runs
            scale = 1.0 / self.dist.world_size
        denc = ws["t"]["denc"].view(N, enc_out.shape[1], enc_out.shape[2], enc_out.shape[3])
        if self.dist is None:
            self.encoder.backward_raw(tuple(img.shape), denc)
        else:
            # encoder buckets: each layer's gradient is all-reduced as soon as its weight-gradient kernels are enqueued (last
            # conv first), small layers coalesced; only the first convs' few kB are left exposed before Adam
            self.encoder.backward_raw(tuple(img.shape), denc, on_layer_grad=self.dist.layer_hook(self.encoder))
            self.dist.wait()
        self._adam(self.decoder.store, scale, self.decoder)
        self._adam(self.encoder.store, scale, self.encoder)
        return ws["t"]["loss"]

    def _keepalive(self):
        """Everything a captured graph replays on (the bounded workspace caches may evict their entries later)."""
        return [list(self.decoder._ws.values()), list(self.encoder._ws.values())]

    def _stores(self):
        """Every flat parameter store the step updates (snapshotted around the pre-capture warm-up steps)."""
        return tuple(getattr(self, n).store for n in ("encoder", "decoder", "row_encoder", "layer2") if getattr(self, n, None) is not None)

    def train_step(self, img, formula, sync=False):
        """img: float tensor [N,1,H,W] (CPU pinned or CUDA); formula: int64 [N,L] (CPU or CUDA).
        Returns the device loss vector [total, ce, reg, n_valid] (no host sync unless sync=True)."""
        N, L = formula.shape
        lengths = torch.full((N, 1), L, dtype=torch.long)                       # img2seq_torch.py:144
        lens, sort_ind = lengths.squeeze(1).sort(dim=0, descending=True)        # seq2seq_torch.py:286 (host, tiny)
        decode_lengths = (lens - 1).tolist()
        img_d = img.to(self.device, non_blocking=True)
        caps_d = formula.to(self.device, non_blocking=True)
        if not torch.equal(sort_ind, torch.arange(N)):
            si = sort_ind.to(self.device)
            img_d, caps_d = img_d[si], caps_d[si]
        T = L - 1
        if not self.use_graph:
            mask = self.decoder.make_dropout_mask(N, T)
            loss = self._step_body(img_d if img_d.dtype == torch.uint8 else img_d.float(), caps_d, decode_lengths, mask)
        else:
            loss = self._graph_step(img_d, caps_d, decode_lengths)
        if sync:
            torch.cuda.synchronize()
        return loss

    def _graph_step(self, img_d, caps_d, decode_lengths):
        frozen = tuple(p_._lo_store_name for m_ in (self.encoder, self.decoder) for p_ in m_.parameters() if not p_.requires_grad)
        key = (tuple(img_d.shape), img_d.dtype, tuple(caps_d.shape), self.decoder.training, frozen)
        g = self._graphs.get(key)
        if g is None:
            N, T = caps_d.shape[0], caps_d.shape[1] - 1
            st = {"img": torch.zeros(img_d.shape, dtype=torch.uint8 if img_d.dtype == torch.uint8 else torch.float32, device=self.device),
                  "caps": torch.zeros(caps_d.shape, dtype=torch.int64, device=self.device)}
            st["img"].copy_(img_d)
            st["caps"].copy_(caps_d)
            # warm-up outside capture (allocates workspaces, sets kernel attributes); it must not train:
            # parameters, Adam moments/step and the bf16 shadows are restored afterwards
            stores = self._stores()
            snap = [{k: getattr(S, k).clone() for k in ("master", "m", "v", "adam_state", "shadow") if getattr(S, k) is not None}
                    for S in stores]
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    mask = self.decoder.make_dropout_mask(N, T)
                    self._step_body(st["img"], st["caps"], decode_lengths, mask)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            for S, sn in zip(stores, snap):
                for k, v in sn.items():
                    getattr(S, k).copy_(v)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                mask = self.decoder.make_dropout_mask(N, T)
                st["loss"] = self._step_body(st["img"], st["caps"], decode_lengths, mask)
            st["graph"] = graph          # capture records the launches, it does not execute them
            # the graph replays on the workspaces that were live during capture: keep them alive even if the bounded
            # workspace caches evict their entries
            st["keep"] = self._keepalive()
            g = self._graphs[key] = st
        g["img"].copy_(img_d, non_blocking=True)
        g["caps"].copy_(caps_d, non_blocking=True)
        g["graph"].replay()
        return g["loss"]

    def getLoss(self, img, formula, lr=None, dropout=None, training=True):
        """img2seq_torch.py:136-172.  Returns -loss as a Python float (one device->host read)."""
        loss = self.train_step(img, formula)
        return -float(loss[0].item())

    # --- epoch loop: img2seq_torch.py:90-134 / base_torch.py:169-206 ------------------------------
    def _run_train_epoch(self, config, train_set, val_set, epoch, lr_schedule):
        from .data import minibatches, pad_batch_formulas, pad_batch_images
        batch_size = config.batch_size
        self.train_mode(True)
        losses = []
        t0 = time.time()
        nimg = 0
        if getattr(self, "_batcher", None) is None:
            from .data import PinnedBatcher
            self._batcher = PinnedBatcher(self._vocab.id_pad, self._vocab.id_end)
        for i, (img, formula) in enumerate(minibatches(train_set, batch_size)):
            # pad_batch_images (utils/image.py:27-44, 255 padding) / pad_batch_formulas (utils/text.py:141-164) straight into pinned
            # staging buffers (one per shape bucket): uint8 pixels [N,1,H,W] (img2seq_torch.py:115-117; conv1 casts on the GPU: 4x
            # less H2D, same values) and int64 ids.  getLoss synchronises on the loss, so a buffer is free again when it returns.
            img = self._batcher.images(img)
            formula = self._batcher.formulas(formula)
            loss_eval = self.getLoss(img, formula=formula, lr=getattr(lr_schedule, "lr", None),
                                     dropout=getattr(config, "dropout", None), training=True)
            losses.append(loss_eval)
            nimg += img.shape[0]
            if lr_schedule is not None:
                lr_schedule.update(batch_no=epoch * ((len(train_set) + batch_size - 1) // batch_size) + i)
        self.last_epoch_stats = {"images_per_s": nimg / max(time.time() - t0, 1e-9), "mean_neg_loss": float(np.mean(losses)) if losses else 0.0}
        score = self.last_epoch_stats["mean_neg_loss"]
        if val_set is not None and self._vocab is not None:
            scores = self.evaluate(config, val_set)                                  # img2seq_torch.py:128-132
            score = scores["perplexity"]
            self.last_epoch_stats.update(scores)
            if lr_schedule is not None:
                lr_schedule.update(score=score)
        return score

    def train(self, config, train_set, val_set, lr_schedule):
        """base_torch.py:169-206 / base.py:95-140: epoch loop, weights saved whenever the epoch score is a new best (>=), early
        stopping through ``lr_schedule.stop_training``.  Resume (base.py:40-47, :107-108): epochs below ``self.startepoch`` —
        set by ``restore_latest()`` from the newest ``model.cpkt-<epoch>`` — are skipped."""
        best_score = None
        for epoch in range(config.n_epochs):
            if epoch < getattr(self, "startepoch", 0):
                continue
            score = self._run_train_epoch(config, train_set, val_set, epoch, lr_schedule)
            if best_score is None or score >= best_score:
                best_score = score
                if self._dir_output is not None:
                    self.save_session(epoch)
            if lr_schedule is not None and getattr(lr_schedule, "stop_training", False):
                break
        return best_score

    # --- inference / evaluation: img2seq.py:198-285 (TF surface) ----------------------------------------
    def _decode_ids(self, images, start_id=None, decoding=None, beam_size=None):
        """Token ids per hypothesis rank: list[n_hyp][N] of id lists (NOT truncated), as ``pred_test.ids`` after the
        reshapes of img2seq.py:236-241 / :265-268."""
        from . import decode
        return self._decode_ids_with(decode.greedy_decode, decode.beam_decode, images, start_id, decoding, beam_size)

    def _decode_ids_with(self, greedy_decode, beam_decode, images, start_id, decoding, beam_size):
        """_decode_ids on the given greedy / beam decode functions (signatures of latex_ocr_b200.decode's)."""
        decoding = decoding or getattr(self._config, "decoding", "greedy")
        end_id = self._vocab.id_end if self._vocab is not None else self._n_tok - 1
        start_id = end_id - 1 if start_id is None else start_id          # default: the PAD id (no START in the torch flavour)
        L = int(getattr(self._config, "max_length_formula", 150))
        self.train_mode(False)
        if decoding == "greedy":
            return [greedy_decode(self, images, start_id, end_id, L).tolist()], end_id
        if decoding != "beam_search" and decoding != "beam":
            raise NotImplementedError("decoding=%r: 'greedy' or 'beam_search' (model.json:13)" % (decoding,))
        beam = int(beam_size or getattr(self._config, "beam_size", 5))
        ids, _ = beam_decode(self, images, start_id, end_id, beam, L,
                             div_gamma=float(getattr(self._config, "div_gamma", 1)),
                             div_prob=float(getattr(self._config, "div_prob", 0)))
        return [ids[:, k].tolist() for k in range(beam)], end_id

    def predict_batch(self, images, start_id=None, decoding=None, beam_size=None):
        """img2seq.py:256-277.  images: tensor [N,1,H,W] (float or uint8) or a list of HxWx1 arrays (padded like
        ``pad_batch_images``).  Returns list[n_hyp][N]: each prediction truncated at END and, when the vocabulary has an
        ``id_to_tok`` table, joined into the formula string like the reference (token-id lists otherwise)."""
        from . import decode
        if not torch.is_tensor(images):
            from .data import pad_batch_images
            images = torch.from_numpy(pad_batch_images(list(images))).permute(0, 3, 1, 2).contiguous()
        hyps, end_id = self._decode_ids(images, start_id, decoding, beam_size)
        rev = getattr(self._vocab, "id_to_tok", None)
        out = []
        for hyp in hyps:
            trunc = decode.truncate_end(hyp, end_id)
            out.append([" ".join(rev[i] for i in p) for p in trunc] if rev is not None else trunc)
        return out

    def predict(self, img):
        """img2seq.py:278-285: one image, one string (or id list) per hypothesis rank."""
        return [hyp[0] for hyp in self.predict_batch([img])]

    def _teacher_forced_ce(self, img, formula_t, lens, start_id):
        """(sum of CE over the real tokens incl. END, number of such tokens) of one padded batch — ``ce_words`` / ``n_words`` of
        img2seq.py:72-75 on the torch-flavour decoder (inputs prefixed with START, targets = tokens then END)."""
        inp = torch.cat([torch.full((formula_t.shape[0], 1), start_id, dtype=torch.int64), formula_t], dim=1)
        enc = self.encoder(img.to(self.device))
        preds, caps, dl, _, _ = self.decoder(enc, inp.to(self.device), lens + 1)
        return self._ce_sum(preds, caps[:, 1:], dl)

    @staticmethod
    def _ce_sum(preds, tgt, dl):
        """(sum of CE, number of tokens) over the first dl[b] steps of each row of the logits preds [B,T,V]."""
        ce_sum, n_tok = 0.0, 0
        for b, n in enumerate(dl):
            lp = torch.log_softmax(preds[b, :n].float(), dim=-1)                 # host-side metric arithmetic (plumbing)
            ce_sum += float(-lp.gather(1, tgt[b, :n].unsqueeze(1)).sum().item())
            n_tok += int(n)
        return ce_sum, n_tok

    def write_prediction(self, config, test_set, start_id=None):
        """img2seq.py:215-254: decodes the whole set, writes ``ref.txt`` / ``hyp_<i>.txt`` under ``config.dir_answers`` through
        ``write_answers`` and returns (files, perplexity) with perplexity = -exp(sum CE / n_words) (negated so that 'higher
        is better' model selection works, :252)."""
        from . import metrics
        from .data import minibatches, pad_batch_formulas, pad_batch_images
        self.train_mode(False)
        end_id, pad_id = self._vocab.id_end, self._vocab.id_pad
        start_id = pad_id if start_id is None else start_id
        refs, hyps = [], None
        ce_words, n_words = 0.0, 0
        for imgs, formulas in minibatches(test_set, config.batch_size):
            img = torch.from_numpy(pad_batch_images(imgs)).permute(0, 3, 1, 2).contiguous()
            formula, length = pad_batch_formulas(formulas, pad_id, end_id)
            ce, n = self._teacher_forced_ce(img, torch.from_numpy(formula.astype(np.int64)),
                                            torch.from_numpy(length.astype(np.int64)).unsqueeze(1), start_id)
            ce_words += ce
            n_words += n
            ids, _ = self._decode_ids(img, start_id)
            if hyps is None:
                hyps = [[] for _ in ids]
            for k, h in enumerate(ids):
                hyps[k] += h
            refs += [list(map(int, f)) for f in formulas]
        rev = getattr(self._vocab, "id_to_tok", None) or {i: str(i) for i in range(self._n_tok)}
        dir_answers = getattr(config, "dir_answers", None) or os.path.join(self._dir_output or ".", "answers") + os.sep
        files = metrics.write_answers(refs, hyps or [[]], rev, dir_answers, end_id)
        perp = -float(np.exp(ce_words / float(max(n_words, 1))))
        return files, perp

    def _run_evaluate(self, config, test_set):
        """img2seq.py:198-213: scores of hypothesis 0 against the references through the answer files."""
        from . import metrics
        files, perp = self.write_prediction(config, test_set)
        scores = metrics.score_files(files[0], files[1])
        scores["perplexity"] = perp
        return scores

    def evaluate(self, config, test_set, start_id=None):
        """base.py:142-160 with the TF path's evaluation semantics (the torch path's own evaluate is broken, SURVEY quirk
        Q6): BLEU-4 / edit distance / exact match of hypothesis 0 + negated perplexity."""
        return self._run_evaluate(config, test_set)

    # --- checkpoints: state_dict round-trips with the reference modules ----------------------------
    def state_dict(self):
        return {"encoder": self.encoder.state_dict(), "decoder": self.decoder.state_dict()}

    def load_state_dict(self, sd):
        self.encoder.load_state_dict(sd["encoder"])
        self.decoder.load_state_dict(sd["decoder"])
        self._graphs.clear()                         # captured steps hold the old bf16 shadows' VALUES only through memory
        self.encoder._shadow_fresh = False           # that stays valid, but force the shadows to be rebuilt from the masters
        self.decoder._shadow_fresh = False

    def save(self, path=None):
        path = path or os.path.join(self._dir_output or ".", "model.pt")
        torch.save({k: {n: t.detach().cpu().contiguous() for n, t in v.items()} for k, v in self.state_dict().items()}, path)
        return path

    def restore(self, path=None, map_location=None):
        """base_torch.py:150-160 (``model_path=None`` -> the default path of ``save()``)."""
        path = path or os.path.join(self._dir_output or ".", "model.pt")
        self.load_state_dict(torch.load(path, map_location=map_location or self.device))

    def auto_restore(self):
        """base_torch.py:146-148: restore the default checkpoint if it exists."""
        path = os.path.join(self._dir_output or ".", "model.pt")
        if os.path.isfile(path):
            self.restore(path)
            return True
        return False

    # TF-style epoch checkpoints (base.py:33-69): ``<dir_output>/model_weights/model.cpkt-<epoch>``, ``max_to_keep=1``,
    # and on start-up the newest one is loaded and its epoch becomes ``startepoch``
    def _dir_model(self):
        return os.path.join(self._dir_output or ".", "model_weights")

    @staticmethod
    def _ckpt_epoch(name):
        idx = name.find("-")                         # base.py:45-46
        try:
            return int(name[idx + 1:].split(".")[0]) if idx >= 0 else None
        except ValueError:
            return None

    def save_session(self, epoch):
        """base.py:60-68 (tf.train.Saver(max_to_keep=1).save(..., global_step=epoch)): parameters AND both Adam states, so a
        resumed run continues the same optimisation."""
        d = self._dir_model()
        os.makedirs(d, exist_ok=True)
        path = os.path.join(d, "model.cpkt-%d" % epoch)
        blob = {"epoch": int(epoch), "state_dict": {k: {n: t.detach().cpu().contiguous() for n, t in v.items()}
                                                    for k, v in self.state_dict().items()}}
        opt = {}
        for name, mod in (("encoder", self.encoder), ("decoder", self.decoder)):
            S = mod.store
            if S.m is not None:
                opt[name] = {"m": S.m.cpu(), "v": S.v.cpu(), "adam_state": S.adam_state.cpu()}
        blob["optimizer"] = opt
        torch.save(blob, path + ".tmp")
        os.replace(path + ".tmp", path)
        for f in os.listdir(d):                      # max_to_keep=1
            if f.startswith("model.cpkt-") and f != os.path.basename(path) and not f.endswith(".tmp"):
                os.remove(os.path.join(d, f))
        return path

    def latest_checkpoint(self):
        d = self._dir_model()
        if not os.path.isdir(d):
            return None
        c = [(self._ckpt_epoch(f), f) for f in os.listdir(d) if f.startswith("model.cpkt-") and not f.endswith(".tmp")]
        c = [x for x in c if x[0] is not None]
        return os.path.join(d, max(c)[1]) if c else None

    def restore_latest(self):
        """base.py:40-47: load the newest epoch checkpoint, set ``startepoch`` to its epoch number (the reference re-runs
        that epoch: ``epoch < startepoch`` skips only the earlier ones).  Returns the epoch or None."""
        self.startepoch = 0
        path = self.latest_checkpoint()
        if path is None:
            return None
        blob = torch.load(path, map_location=self.device)
        self.load_state_dict(blob["state_dict"])
        for name, mod in (("encoder", self.encoder), ("decoder", self.decoder)):
            o = blob.get("optimizer", {}).get(name)
            if o is not None:
                S = mod.store
                S.ensure_adam(self.lr)
                S.m.copy_(o["m"])
                S.v.copy_(o["v"])
                S.adam_state.copy_(o["adam_state"])
        self.startepoch = int(blob["epoch"])
        return self.startepoch
