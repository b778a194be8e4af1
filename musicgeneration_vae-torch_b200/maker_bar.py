"""Sampling loop with the semantics of the reference's maker_bar.py:32-44, batched over S independent songs.

Per phrase index the phrase encoder runs ONCE (its input is constant across the 4 inner bar iterations; the
reference recomputes it 4x), each bar is thresholded at 0.3 on the device, and the 4 bars of a phrase become the next
``pre_phrase``.  Songs are independent, so S songs advance in lock-step as one batch (BASELINE config 5: S = 8192).

Two extensions, both off by default: ``sampler="bernoulli"`` draws every cell from the decoder's own Bernoulli
distribution at a temperature instead of thresholding it (csrc/sample.cu), and ``primer`` continues given phrases
instead of starting from silence."""
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


def load_primer(path, music_length, phrases=None):
    """Read a MIDI file as a primer for ``sample_songs``: ``(roll [P*384, 60] float32 {0,1}, P, dropped)``.  The file
    goes through ``midi.midi_to_roll``; notes outside the 60-pitch window (27..86) are dropped and counted.  ``phrases``
    defaults to the whole 384-step phrases the file's notes cover (a partial last phrase is not used); either way
    1 <= P < music_length is required."""
    from .midi import LOWEST_PITCH, N_PITCHES, midi_to_roll, read_midi
    division, _, notes = read_midi(path)
    dropped = sum(1 for p, _, _, _ in notes if not LOWEST_PITCH <= p < LOWEST_PITCH + N_PITCHES)
    if phrases is None:
        from .midi import BEAT_RESOLUTION
        steps = max((e * BEAT_RESOLUTION // division for _, _, e, _ in notes), default=0)
        phrases = steps // PHRASE_STEPS
        if phrases == 0:
            raise ValueError("primer %s covers no whole %d-step phrase" % (path, PHRASE_STEPS))
    if not 1 <= phrases < music_length:
        raise ValueError("primer: %d phrases; need 1 <= P < music_length = %d" % (phrases, music_length))
    roll = midi_to_roll(path, phrases * PHRASE_STEPS)
    check_primer(roll, 1, music_length)
    return roll, phrases, dropped


def main(argv=None):
    """The reference script (maker_bar.py:10-54): load ``model/checkpoint_{model_number}.pth.tar``, sample
    ``music_length`` phrases of 4 bars, write ``./test.mid``.  ``--sampler bernoulli`` draws the cells at
    ``--temperature`` instead of thresholding them; ``--primer x.mid`` continues the file's first phrases (all songs
    continue the same primer).  ``--seed`` seeds both the latents and the Bernoulli stream."""
    import argparse
    import math
    from .graph.model import Model
    from .midi import write_midi
    ap = argparse.ArgumentParser()
    ap.add_argument("--model_number", type=int, default=10, help="Music length that want to make.")
    ap.add_argument("--music_length", type=int, default=10, help="Music length that want to make.")
    ap.add_argument("--songs", type=int, default=1, help="independent songs sampled in lock-step (test_<i>.mid)")
    ap.add_argument("--out", default="./test.mid")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--sampler", choices=SAMPLERS, default="threshold",
                    help="threshold: cell = prob > 0.3 (the reference); bernoulli: draw each cell at --temperature")
    ap.add_argument("--temperature", type=float, default=1.0, help="Bernoulli sampler: logits are divided by it")
    ap.add_argument("--primer", default=None, help="MIDI file whose first phrases the songs continue")
    ap.add_argument("--primer_phrases", type=int, default=None,
                    help="phrases of the primer to use (default: the whole phrases the file covers)")
    args = ap.parse_args(argv)
    if not (math.isfinite(args.temperature) and args.temperature > 0):
        ap.error("--temperature must be finite and > 0")
    if args.primer_phrases is not None and args.primer is None:
        ap.error("--primer_phrases needs --primer")
    primer = None
    if args.primer is not None:
        try:
            primer, P, dropped = load_primer(args.primer, args.music_length, args.primer_phrases)
        except ValueError as e:
            ap.error(str(e))
        print("primer: %d phrases from %s, %d notes outside pitches 27..86 dropped" % (P, args.primer, dropped))
    dev = torch.device("cuda", torch.cuda.current_device())
    model = load_generator(Model().to(dev), "model/checkpoint_{}.pth.tar".format(args.model_number), dev)
    g = torch.Generator(device=dev)
    if args.seed is not None:
        g.manual_seed(args.seed)
    seed = g.initial_seed()
    print("seed:", seed)
    lat = torch.randn(args.music_length * 4, args.songs, 1152, device=dev, generator=g)
    if primer is not None:
        primer = torch.from_numpy(primer).to(dev)
    rolls = songs_to_host(sample_songs(model, lat, args.music_length, sampler=args.sampler,
                                       temperature=args.temperature, seed=seed, primer=primer))
    for i, r in enumerate(rolls):
        path = args.out if i == 0 else args.out.replace(".mid", "_%d.mid" % i)
        print(r.shape, write_midi(r, path), "notes ->", path)


if __name__ == "__main__":
    main()
