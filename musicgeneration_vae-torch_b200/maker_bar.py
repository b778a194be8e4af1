"""Sampling loop with the semantics of the reference's maker_bar.py:32-44, batched over S independent songs.

Per phrase index the phrase encoder runs ONCE (its input is constant across the 4 inner bar iterations; the
reference recomputes it 4x), each bar is thresholded at 0.3 on the device, and the 4 bars of a phrase become the next
``pre_phrase``.  Songs are independent, so S songs advance in lock-step as one batch (BASELINE config 5: S = 8192).

Two extensions, both off by default: ``sampler="bernoulli"`` draws every cell from the decoder's own Bernoulli
distribution at a temperature instead of thresholding it (csrc/sample.cu), and ``primer`` continues given phrases
instead of starting from silence."""
import collections
import itertools
import math
import os

import numpy as np
import torch

PHRASE_STEPS, PITCHES = 384, 60
SAMPLERS = ("threshold", "bernoulli")


def check_primer(primer, songs, music_length):
    """Validate a primer for ``sample_songs``: ``[songs, P*384, 60]`` or ``[P*384, 60]`` (one primer for every song),
    {0,1} cells, 1 <= P < music_length whole phrases.  Returns P.  Runs wherever the tensor lives (no device needed)."""
    shape = tuple(primer.shape)
    if len(shape) not in (2, 3) or shape[-1] != PITCHES or (len(shape) == 3 and shape[0] != songs):
        raise ValueError("primer: expected shape [%d, P*%d, %d] or [P*%d, %d], got %r"
                         % (songs, PHRASE_STEPS, PITCHES, PHRASE_STEPS, PITCHES, shape))
    steps = shape[-2]
    if steps % PHRASE_STEPS:
        raise ValueError("primer: %d time steps is not a whole number of %d-step phrases" % (steps, PHRASE_STEPS))
    P = steps // PHRASE_STEPS
    if not 1 <= P < music_length:
        raise ValueError("primer: %d phrases; need 1 <= P < music_length = %d" % (P, music_length))
    t = primer if isinstance(primer, torch.Tensor) else torch.as_tensor(np.asarray(primer))
    if not bool(((t == 0) | (t == 1)).all()):
        raise ValueError("primer: cells must be exactly 0 or 1")
    return P


@torch.no_grad()
def sample_songs(model, latents, music_length, return_first_probs=False, threshold=0.3, *,
                 sampler="threshold", temperature=1.0, seed=0, song_base=0, primer=None):
    """latents: [music_length*4, S, 1152] (the randn draws, one per bar).  Returns uint8-valued float piano-roll
    [S, music_length*4*96, 60] (and optionally the first generated bar's probabilities).

    ``sampler="threshold"``: cell = prob > ``threshold`` (maker_bar.py:39); ``temperature``, ``seed`` and
    ``song_base`` have no effect.  ``sampler="bernoulli"``: cell ~ Bernoulli(sigmoid(logit / temperature)), drawn by
    ``data.packed.bernoulli_sample`` from the stream of (``seed``, song ``song_base + s``, bar ``k``, cell), so a song is
    the same whatever batch it is sampled in.  Not available with ``Model(refiner=True)`` (the Refiner outputs
    probabilities, not logits).

    ``primer``: P whole phrases of {0,1} cells, ``[S, P*384, 60]`` or ``[P*384, 60]`` for all songs, 1 <= P <
    music_length.  They are the first P phrases of the output, verbatim; generation starts at phrase P with the
    primer's last bar as ``pre_bar``, its last phrase as ``pre_phrase`` and the position ``phrase_idx[P]``.  Bar k
    always uses ``latents[k]`` (the primer's latents are unused), so a primed run continues exactly as the unprimed run
    that produced the primer would have, for the same latents and seed."""
    if sampler not in SAMPLERS:
        raise ValueError("sample_songs: sampler must be one of %s, got %r" % (SAMPLERS, sampler))
    bernoulli = sampler == "bernoulli"
    if bernoulli:
        if getattr(model, "refiner", None) is not None:
            raise ValueError("sample_songs: sampler='bernoulli' needs the decoder's logits; Model(refiner=True) "
                             "outputs probabilities")
        from .data.packed import bernoulli_sample
    S = latents.shape[1]
    dev = latents.device
    P = 0 if primer is None else check_primer(primer, S, music_length)
    pre_phrase = torch.zeros(S, 1, 384, 60, device=dev)
    pre_bar = torch.zeros(S, 1, 96, 60, device=dev)
    phrase_idx = [330] + [i for i in range(music_length - 2, -1, -1)]     # maker_bar.py:34
    out = torch.empty(S, music_length * 4, 96, 60, device=dev)
    if P:
        prim = torch.as_tensor(primer).to(device=dev, dtype=torch.float32)
        out[:, :4 * P] = prim.reshape(-1, 4 * P, 96, 60).expand(S, -1, -1, -1)
        pre_bar = out[:, 4 * P - 1:4 * P].clone()
        pre_phrase = out[:, 4 * P - 4:4 * P].reshape(S, 1, 384, 60)
    was_training = model.training
    model.eval()
    first = None
    k = 4 * P
    for idx in range(P, music_length):
        pos = torch.full((S,), phrase_idx[idx], dtype=torch.long, device=dev)
        phrase_feature = model.phrase_encoder(pre_phrase)               # once per phrase
        for _ in range(4):
            pre_z = model.encoder(pre_bar)
            if bernoulli:
                probs, logits = model.decoder.forward_logits(latents[k], pre_z, phrase_feature, pos)
            else:
                probs = model.decoder(latents[k], pre_z, phrase_feature, pos)
                if getattr(model, "refiner", None) is not None:
                    probs = model.refiner(probs)                         # graph/model.py:41 (Model(refiner=True))
            if first is None:
                first = probs.clone()
            if bernoulli:
                pre_bar = bernoulli_sample(logits, temperature, seed, song_base, k)
            else:
                pre_bar = (probs > threshold).float()                    # maker_bar.py:39
            out[:, k] = pre_bar[:, 0]
            k += 1
        pre_phrase = out[:, k - 4:k].reshape(S, 1, 384, 60)
    model.train(was_training)
    roll = out.reshape(S, music_length * 4 * 96, 60)
    return (roll, first) if return_first_probs else roll


# ---- songs -> latents: encoding, teacher-forced reconstruction, interpolation ------------------------------------------
Reconstruction = collections.namedtuple("Reconstruction", "latents nll counts logits")
SLERP_EPS = 1e-4        # radians: below this angle (or within it of pi) interpolate_latents is linear


def _song_roll(roll, device):
    """``[S, L*384, 60]`` or ``[L*384, 60]`` {0,1} cells, L >= 1 -> (contiguous fp32 [S, 4L, 96, 60] on ``device``,
    S, L)"""
    t = torch.as_tensor(roll)
    shape = tuple(t.shape)
    if (len(shape) not in (2, 3) or shape[-1] != PITCHES or shape[-2] == 0 or shape[-2] % PHRASE_STEPS
            or (len(shape) == 3 and shape[0] == 0)):
        raise ValueError("roll: expected shape [S, L*%d, %d] or [L*%d, %d] with L >= 1 whole phrases, got %r"
                         % (PHRASE_STEPS, PITCHES, PHRASE_STEPS, PITCHES, shape))
    t = t.to(device=device, dtype=torch.float32).contiguous()
    if not bool(((t == 0) | (t == 1)).all()):
        raise ValueError("roll: cells must be exactly 0 or 1")
    L = shape[-2] // PHRASE_STEPS
    return t.view(-1, 4 * L, 96, PITCHES), t.numel() // (L * PHRASE_STEPS * PITCHES), L


def _encode_all(trunk, items, chunk, zero_first=False):
    """``trunk.encode`` over ``items`` [N, H, W] (preceded by one all-zero item if ``zero_first``) in passes of at most
    ``chunk`` items; -> [N (+1), 1152] fp32.  Each pass's input is built in bf16, the trunk's input type, so the
    leading zero item costs no extra copy of the roll."""
    lead = int(zero_first)
    n = items.shape[0] + lead
    out = torch.empty(n, 1152, device=items.device)
    for i in range(0, n, chunk):
        j = min(n, i + chunk)
        x = torch.empty((j - i, 1) + tuple(items.shape[1:]), dtype=torch.bfloat16, device=items.device)
        if i < lead:
            x[0].zero_()
        x[max(lead - i, 0):, 0].copy_(items[max(i - lead, 0):j - lead])
        out[i:j] = trunk.encode(x)
    return out


def _check_chunk(chunk):
    if int(chunk) < 1:
        raise ValueError("chunk must be >= 1 (got %r)" % (chunk,))
    return int(chunk)


@torch.no_grad()
def encode_songs(model, roll, chunk=8192):
    """The latents of whole songs: ``roll`` [S, L*384, 60] or [L*384, 60] (one song) of {0,1} cells, L >= 1 phrases
    -> [4L, S, 1152] fp32, ``latents[k, s] = model.encoder(bar k of song s)``: the ``z`` of training, and the layout
    ``sample_songs`` takes.  With ``Model(vae_head=True)`` this is the posterior mean (the encoder is the mean head).
    Every bar is encoded once, in passes of at most ``chunk`` bars, in inference mode."""
    chunk = _check_chunk(chunk)
    bars, S, L = _song_roll(roll, next(model.parameters()).device)
    z = _encode_all(model.encoder, bars.view(-1, 96, PITCHES), chunk)
    return z.view(S, 4 * L, 1152).transpose(0, 1).contiguous()


@torch.no_grad()
def reconstruct_songs(model, roll, temperature=1.0, threshold=0.3, chunk=8192, return_logits=False):
    """Teacher-forced pass over whole songs (``roll`` as for ``encode_songs``): every bar is decoded from its own
    latent with the conditioning ``sample_songs`` gives a song of L phrases -- bar k of phrase p = k // 4 from
    ``z = encoder(bar k)``, ``pre_z = encoder(bar k-1)`` (of the zero bar for k = 0), the phrase feature of phrase p-1
    (of the zero phrase for p = 0) and the position ``phrase_idx[p]`` -- and scored by ``data.packed.score_bars``
    against the bar itself under Bernoulli(sigmoid(logit / ``temperature``)).

    Every input is known in advance, so all S*4L bars run as one batched encoder pass (plus the zero bar), one phrase
    encoder pass over the S*(L-1) conditioning phrases (plus the zero phrase) and one decoder pass, each in passes of at
    most ``chunk`` bars (``chunk // 4`` phrases), instead of 4L dependent bar steps.

    Returns ``Reconstruction(latents [4L, S, 1152] (as encode_songs), nll [S, 4L] fp32 nats, counts [S, 4L, 3] int32
    (cells with p > threshold that are on, cells with p > threshold, cells on), logits [S, 4L, 96, 60] or None)``; the
    logits (23 KB per bar) only with ``return_logits``.  With ``Model(vae_head=True)`` the latents are the posterior
    means.  Not available with ``Model(refiner=True)``: the Refiner outputs probabilities, not logits."""
    from .data.packed import score_bars
    if getattr(model, "refiner", None) is not None:
        raise ValueError("reconstruct_songs needs the decoder's logits; Model(refiner=True) outputs probabilities")
    chunk = _check_chunk(chunk)
    dev = next(model.parameters()).device
    bars, S, L = _song_roll(roll, dev)
    K, N = 4 * L, S * 4 * L
    was_training = model.training
    model.eval()
    try:
        zz = _encode_all(model.encoder, bars.view(N, 96, PITCHES), chunk, zero_first=True)     # [zero bar, bars]
        phrases = bars.view(S, L, 4 * 96, PITCHES)[:, :L - 1].reshape(S * (L - 1), 4 * 96, PITCHES)
        pf = _encode_all(model.phrase_encoder.phrase_encoder, phrases, max(1, chunk // 4), zero_first=True)
        # row r = s*K + k: z = zz[1 + r], pre_z = zz[r] (zz[0] for k = 0), phrase p = k // 4 -> pf[0] for p = 0, else
        # pf[1 + s*(L-1) + p-1]
        r = torch.arange(N, device=dev)
        s, k = r // K, r % K
        p = k // 4
        pre_idx = torch.where(k == 0, 0, r)
        pf_idx = torch.where(p == 0, 0, 1 + s * (L - 1) + p - 1)
        phrase_idx = torch.tensor([330] + list(range(L - 2, -1, -1)), device=dev)       # maker_bar.py:34
        pos = phrase_idx[p]
        nll = torch.empty(N, device=dev)
        counts = torch.empty(N, 3, dtype=torch.int32, device=dev)
        logits = torch.empty(N, 96, PITCHES, device=dev) if return_logits else None
        target = bars.view(N, 96, PITCHES)
        for i in range(0, N, chunk):
            j = min(N, i + chunk)
            _, lg = model.decoder.forward_logits(zz[1 + i:1 + j], zz.index_select(0, pre_idx[i:j]),
                                                 pf.index_select(0, pf_idx[i:j]), pos[i:j])
            nll[i:j], counts[i:j] = score_bars(lg, target[i:j], temperature, threshold)
            if logits is not None:
                logits[i:j] = lg.view(j - i, 96, PITCHES)
    finally:
        model.train(was_training)
    return Reconstruction(zz[1:].view(S, K, 1152).transpose(0, 1).contiguous(), nll.view(S, K),
                          counts.view(S, K, 3), None if logits is None else logits.view(S, K, 96, PITCHES))


def interpolate_latents(za, zb, steps):
    """Morph one song's latents into another's: ``za``, ``zb`` [K, 1152] or [K, 1, 1152] (``encode_songs`` of one
    song) -> [K, steps, 1152], point i at t = i / (steps - 1) of the spherical interpolation of every bar vector,
    computed in float64 and returned in ``za``'s dtype.  Where either vector is zero, or the angle between them is
    below ``SLERP_EPS`` radians or within it of pi (no unique great circle), the interpolation is linear.  Point 0 is
    exactly ``za`` and point steps-1 exactly ``zb``.  Each point is one song of a ``sample_songs`` batch, so a morph
    decodes in lock-step with either sampler.  Plain PyTorch; runs on CPU tensors too."""
    if int(steps) != steps or steps < 2:
        raise ValueError("interpolate_latents: steps must be an integer >= 2 (got %r)" % (steps,))
    steps = int(steps)
    if za.shape != zb.shape or za.dim() not in (2, 3) or (za.dim() == 3 and za.shape[1] != 1):
        raise ValueError("interpolate_latents: za and zb must both be [K, D] or [K, 1, D], got %r and %r"
                         % (tuple(za.shape), tuple(zb.shape)))
    a = za.reshape(za.shape[0], 1, -1)
    b = zb.reshape(zb.shape[0], 1, -1).to(a.device)
    a64, b64 = a.double(), b.double()
    t = (torch.arange(steps, dtype=torch.float64, device=a.device) / (steps - 1)).view(1, -1, 1)
    na, nb = a64.norm(dim=-1, keepdim=True), b64.norm(dim=-1, keepdim=True)
    cos = ((a64 * b64).sum(-1, keepdim=True) / (na * nb).clamp_min(1e-300)).clamp(-1.0, 1.0)
    omega = torch.acos(cos)
    sin = torch.sin(omega)
    linear = (na == 0) | (nb == 0) | (omega < SLERP_EPS) | (omega > math.pi - SLERP_EPS)
    safe = torch.where(linear, torch.ones_like(sin), sin)
    wa = torch.where(linear, 1.0 - t, torch.sin((1.0 - t) * omega) / safe)
    wb = torch.where(linear, t, torch.sin(t * omega) / safe)
    out = (wa * a64 + wb * b64).to(za.dtype)
    out[:, 0] = a[:, 0]
    out[:, -1] = b[:, 0]
    return out


def songs_to_host(roll):
    """Device roll [S, T, 60] of {0,1} floats -> numpy float32 on the host, crossing PCIe as bits: one
    bvae_threshold_pack launch (720 B per bar instead of the 23 KB the reference reads back per bar at
    maker_bar.py:40), expanded again with numpy on the host."""
    from .data.packed import threshold_pack, unpack_cells_host
    bits, _ = threshold_pack(roll, 0.5)
    return unpack_cells_host(bits.cpu().numpy(), tuple(roll.shape))


def load_generator(model, filename, device="cuda"):
    """maker_bar.py:25-30: ``checkpoint['generator_state_dict']`` saved from nn.DataParallel (``module.`` prefix); the
    reference's Refiner entries are ignored (graph/refiner.py cannot execute, SURVEY.md section 0)."""
    ck = torch.load(filename, map_location=device, weights_only=False)
    sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in ck["generator_state_dict"].items()}
    own = model.state_dict()
    # Refiner entries load only into Model(refiner=True), and only where the shapes agree: the reference's
    # refiner.layer2.0.weight [8,1,4,4] IS its defect (graph/refiner.py:19)
    sd = {k: v for k, v in sd.items() if not k.startswith("refiner.") or (k in own and tuple(own[k].shape) == tuple(v.shape))}
    model.load_state_dict(sd, strict=False)
    return model


def load_roll(path, phrases=None):
    """Read a MIDI file as a piano-roll: ``(roll [P*384, 60] float32 {0,1}, P, dropped)``.  The file goes through
    ``midi.midi_to_roll``; notes outside the 60-pitch window (27..86) are dropped and counted.  ``phrases`` defaults to
    the whole 384-step phrases the file's notes cover (a partial last phrase is not used; P = 0 when there is none);
    an explicit ``phrases`` beyond the notes gives silent phrases."""
    from .midi import BEAT_RESOLUTION, LOWEST_PITCH, N_PITCHES, midi_to_roll, read_midi
    division, _, notes = read_midi(path)
    dropped = sum(1 for p, _, _, _ in notes if not LOWEST_PITCH <= p < LOWEST_PITCH + N_PITCHES)
    if phrases is None:
        steps = max((e * BEAT_RESOLUTION // division for _, _, e, _ in notes), default=0)
        phrases = steps // PHRASE_STEPS
    elif phrases < 0:
        raise ValueError("load_roll: phrases must be >= 0 (got %d)" % phrases)
    return midi_to_roll(path, phrases * PHRASE_STEPS), phrases, dropped


def load_primer(path, music_length, phrases=None):
    """Read a MIDI file as a primer for ``sample_songs``: ``(roll [P*384, 60] float32 {0,1}, P, dropped)`` from
    ``load_roll``.  ``phrases`` defaults to the whole 384-step phrases the file's notes cover; either way
    1 <= P < music_length is required."""
    if phrases is not None and not 1 <= phrases < music_length:
        raise ValueError("primer: %d phrases; need 1 <= P < music_length = %d" % (phrases, music_length))
    roll, phrases, dropped = load_roll(path, phrases)
    if phrases == 0:
        raise ValueError("primer %s covers no whole %d-step phrase" % (path, PHRASE_STEPS))
    if not 1 <= phrases < music_length:
        raise ValueError("primer: %d phrases; need 1 <= P < music_length = %d" % (phrases, music_length))
    check_primer(roll, 1, music_length)
    return roll, phrases, dropped


def score_line(rec, threshold=0.3, temperature=1.0):
    """One line summarising a ``Reconstruction``: mean NLL per bar, cells on, precision / recall / F1 at ``threshold``"""
    tp, on, pos = (int(v) for v in rec.counts.sum((0, 1), dtype=torch.int64).tolist())
    precision = tp / on if on else 0.0
    recall = tp / pos if pos else 0.0
    f1 = 2 * precision * recall / (precision + recall) if precision + recall else 0.0
    return ("teacher-forced score: nll %.6f nats/bar over %d bars (T=%g), cells on %d, predicted on %d, "
            "precision %.6f recall %.6f f1 %.6f at %g" % (float(rec.nll.double().mean()), rec.nll.numel(), temperature,
                                                          pos, on, precision, recall, f1, threshold))


def main(argv=None):
    """The reference script (maker_bar.py:10-54): load ``model/checkpoint_{model_number}.pth.tar``, sample
    ``music_length`` phrases of 4 bars, write ``./test.mid``.  ``--sampler bernoulli`` draws the cells at
    ``--temperature`` instead of thresholding them; ``--primer x.mid`` continues the file's first phrases (all songs
    continue the same primer).  ``--seed`` seeds both the latents and the Bernoulli stream.

    ``--reconstruct x.mid`` encodes the file's whole phrases (``--phrases N``: the first N), writes the free-running
    decode of those latents to ``--out`` and prints the teacher-forced score.  ``--interpolate a.mid b.mid`` encodes
    both files, cut to the same number of whole phrases (the smaller count, or ``--phrases``), and writes ``--steps``
    songs morphing from a to b: ``--out``, ``out_1``, ...  In both modes the song length is the file's, not
    ``--music_length``.

    ``--fit_prior OUT.pt --data SRC [SRC ...]`` fits a Gaussian to the checkpoint's latents of every bar of the sources
    (``.mid`` files, whole phrases, or packed-array directories of ``tools/pack_dataset.py``), writes it to ``OUT.pt``
    and samples nothing.  ``--latent_prior PRIOR.pt`` then draws the latents of the default and ``--primer`` modes from
    that prior instead of N(0, I) (prior.py); a prior fitted to another checkpoint is refused."""
    import argparse
    from .graph.model import Model
    from .midi import write_midi
    ap = argparse.ArgumentParser()
    ap.add_argument("--model_number", type=int, default=10, help="Music length that want to make.")
    ap.add_argument("--music_length", type=int, default=10, help="Music length that want to make.")
    ap.add_argument("--songs", type=int, default=None,
                    help="independent songs sampled in lock-step (test_<i>.mid); default 1")
    ap.add_argument("--out", default="./test.mid")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--sampler", choices=SAMPLERS, default="threshold",
                    help="threshold: cell = prob > 0.3 (the reference); bernoulli: draw each cell at --temperature")
    ap.add_argument("--temperature", type=float, default=1.0, help="Bernoulli sampler: logits are divided by it")
    ap.add_argument("--primer", default=None, help="MIDI file whose first phrases the songs continue")
    ap.add_argument("--primer_phrases", type=int, default=None,
                    help="phrases of the primer to use (default: the whole phrases the file covers)")
    ap.add_argument("--reconstruct", default=None, metavar="X.MID",
                    help="encode the file, write the decode of its latents, print the teacher-forced score")
    ap.add_argument("--interpolate", nargs=2, default=None, metavar=("A.MID", "B.MID"),
                    help="write --steps songs morphing from A to B through the latent space")
    ap.add_argument("--steps", type=int, default=None, help="--interpolate: songs from A to B, >= 2 (default 5)")
    ap.add_argument("--phrases", type=int, default=None,
                    help="--reconstruct / --interpolate: phrases of the file(s) to use (default: the whole phrases "
                         "covered; for two files the smaller count)")
    ap.add_argument("--latent_prior", default=None, metavar="PRIOR.pt",
                    help="draw the latents from this fitted prior (--fit_prior) instead of N(0, I)")
    ap.add_argument("--fit_prior", default=None, metavar="OUT.pt",
                    help="fit a Gaussian prior to the checkpoint's latents of the --data bars, write it, sample nothing")
    ap.add_argument("--data", nargs="+", default=None, metavar="SRC",
                    help="--fit_prior: .mid files and packed-array directories (tools/pack_dataset.py) to fit on")
    args = ap.parse_args(argv)
    if not (math.isfinite(args.temperature) and args.temperature > 0):
        ap.error("--temperature must be finite and > 0")
    if args.primer_phrases is not None and args.primer is None:
        ap.error("--primer_phrases needs --primer")
    modes = [m for m in ("primer", "reconstruct", "interpolate") if getattr(args, m) is not None]
    if len(modes) > 1:
        ap.error("--primer, --reconstruct and --interpolate are mutually exclusive")
    encode_mode = modes[0] if modes and modes[0] != "primer" else None
    if encode_mode and args.songs is not None:
        ap.error("--songs does not apply to --%s" % encode_mode)
    if args.steps is not None and encode_mode != "interpolate":
        ap.error("--steps needs --interpolate")
    if args.steps is not None and args.steps < 2:
        ap.error("--steps must be at least 2")
    if args.phrases is not None and not encode_mode:
        ap.error("--phrases needs --reconstruct or --interpolate")
    if args.phrases is not None and args.phrases < 1:
        ap.error("--phrases must be at least 1")
    if args.latent_prior is not None and encode_mode:
        ap.error("--latent_prior does not apply to --%s" % encode_mode)
    if args.fit_prior is not None:
        if modes or args.latent_prior is not None:
            ap.error("--fit_prior does not combine with --%s" % (modes[0] if modes else "latent_prior"))
        if args.songs is not None:
            ap.error("--songs does not apply to --fit_prior")
        if args.data is None:
            ap.error("--fit_prior needs --data")
        for src in args.data:
            if not (os.path.isfile(os.path.join(src, "note_bits.npy")) or
                    (os.path.isfile(src) and src.lower().endswith((".mid", ".midi")))):
                ap.error("--data %s is neither a .mid file nor a packed-array directory with note_bits.npy" % src)
    elif args.data is not None:
        ap.error("--data needs --fit_prior")
    if args.latent_prior is not None and not os.path.isfile(args.latent_prior):
        ap.error("--latent_prior %s: no such file" % args.latent_prior)
    primer = None
    if args.primer is not None:
        try:
            primer, P, dropped = load_primer(args.primer, args.music_length, args.primer_phrases)
        except ValueError as e:
            ap.error(str(e))
        print("primer: %d phrases from %s, %d notes outside pitches 27..86 dropped" % (P, args.primer, dropped))
    rolls_in = []
    for path in ([args.reconstruct] if encode_mode == "reconstruct" else args.interpolate or []):
        roll, P, dropped = load_roll(path, args.phrases)
        if P == 0:
            ap.error("%s covers no whole %d-step phrase" % (path, PHRASE_STEPS))
        print("%s: %d phrases from %s, %d notes outside pitches 27..86 dropped" % (encode_mode, P, path, dropped))
        rolls_in.append(roll)
    if rolls_in:
        P = min(r.shape[0] for r in rolls_in) // PHRASE_STEPS
        rolls_in = np.stack([r[:P * PHRASE_STEPS] for r in rolls_in])
    dev = torch.device("cuda", torch.cuda.current_device())
    model = load_generator(Model().to(dev), "model/checkpoint_{}.pth.tar".format(args.model_number), dev)
    if args.fit_prior is not None:
        from .prior import bars_of_midi, bars_of_packed, fit_latent_prior, save_latent_prior
        srcs = [bars_of_packed(src) if os.path.isdir(src) else bars_of_midi([src]) for src in args.data]
        try:
            prior = fit_latent_prior(model, itertools.chain.from_iterable(srcs))
        except ValueError as e:
            ap.error(str(e))
        save_latent_prior(prior, args.fit_prior)
        print("latent prior: %d bars, |mean| %.6g, sqrt(trace(cov) / d) %.6g, shrinkage %g -> %s"
              % (prior.count, float(prior.mean.norm()), math.sqrt(float(torch.trace(prior.cov)) / prior.dim),
                 prior.shrinkage, args.fit_prior))
        return
    prior = None
    if args.latent_prior is not None:
        from .prior import load_latent_prior
        try:
            prior = load_latent_prior(args.latent_prior, model)
        except ValueError as e:
            ap.error(str(e))
    g = torch.Generator(device=dev)
    if args.seed is not None:
        g.manual_seed(args.seed)
    seed = g.initial_seed()
    print("seed:", seed)
    length = args.music_length
    if encode_mode == "reconstruct":
        rec = reconstruct_songs(model, rolls_in[0], temperature=args.temperature)
        print(score_line(rec, temperature=args.temperature))
        lat, length = rec.latents, P
    elif encode_mode == "interpolate":
        z = encode_songs(model, rolls_in)
        lat, length = interpolate_latents(z[:, 0], z[:, 1], 5 if args.steps is None else args.steps), P
    elif prior is not None:
        lat = prior.sample(args.music_length * 4, 1 if args.songs is None else args.songs, g)
    else:
        lat = torch.randn(args.music_length * 4, 1 if args.songs is None else args.songs, 1152, device=dev,
                          generator=g)
    if primer is not None:
        primer = torch.from_numpy(primer).to(dev)
    rolls = songs_to_host(sample_songs(model, lat, length, sampler=args.sampler,
                                       temperature=args.temperature, seed=seed, primer=primer))
    for i, r in enumerate(rolls):
        path = args.out if i == 0 else args.out.replace(".mid", "_%d.mid" % i)
        print(r.shape, write_midi(r, path), "notes ->", path)


if __name__ == "__main__":
    main()
