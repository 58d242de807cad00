"""Entry point mirroring postprocessing/decoding.py:6-53."""
import torch


def decode(model, input, data_loader=None, expected=None, method="greedy", beam_width=3, stop_at_eos=False):
    """Same arguments, return value and error behaviour as the reference's
    ``decode``: greedy -> int64 [B, expected.size(1)-1] on the input's device
    (logits -> transpose -> topk(1) over the vocab axis, decoding.py:35-40);
    beam -> int64 [B, expected.size(-1)-1] on the CPU (decoding.py:42-48).

    ``stop_at_eos`` (greedy only; beam search stops at <EOS> already): decode each image only up to its first <EOS>
    and return <PAD> after it -- the same strings from id_to_string (utils/utils.py:134-164), less decoder work."""
    if method == "greedy" and stop_at_eos:
        _, sequence, _ = model.greedy_until_eos(input, expected.size(1) - 1)
    elif method == "greedy":
        output = model(input=input, expected=expected, is_train=False, teacher_forcing_ratio=0.0)
        decoded_values = output.transpose(1, 2)
        _, sequence = torch.topk(decoded_values, 1, dim=1)
        sequence = sequence.squeeze(1)
    elif method == "beam":
        sequence = model.beam_search(input=input, data_loader=data_loader, beam_width=beam_width,
                                     max_sequence=expected.size(-1) - 1)
    else:
        raise NotImplementedError(f"There's no '{method}' type yet.")
    return sequence


RULE_BITS = ("cannot_initial", "next_underbar", "next_lbracket", "cannot_next_underbar", "cannot_next_lbracket")


def compile_decoding_rules(manager):
    """Per-class tables for ``frx_set_decoding_rules`` from a reference-style DecodingManager
    (postprocessing/postprocessing.py:182-191: ``.rules`` is the RULES dict, ``.tokens`` the 245 class names).

    Returns (flags, limit, ids6) as Python int lists: flags bit i <-> ``rules[RULE_BITS[i]]`` contains the token;
    limit[v] = ``limit_params[token]`` where ``limit_series[token]`` is true (MemoryNode._look_back, :327-391);
    ids6 = ids of "<SOS>", "<EOS>", "" (the empty class), "{", "}", "_"."""
    tokens = list(manager.tokens)
    index = {t: i for i, t in enumerate(tokens)}
    flags, limit = [0] * len(tokens), [0] * len(tokens)
    for bit, key in enumerate(RULE_BITS):
        for t in manager.rules.get(key, ()):
            if t not in index:
                raise KeyError("decoding rule %r names the unknown token %r" % (key, t))
            flags[index[t]] |= 1 << bit
    series, params = manager.rules.get("limit_series", {}), manager.rules.get("limit_params", {})
    for t, on in series.items():
        if on and t in index:
            if t not in params:
                raise KeyError("limit_series enables %r but limit_params has no entry for it" % t)
            limit[index[t]] = int(params[t])
    ids6 = [index[t] for t in ("<SOS>", "<EOS>", "", "{", "}", "_")]
    return flags, limit, ids6
