"""Deterministic synthetic inputs of the shapes BASELINE.json names (SURVEY.md section 8(d)).

No corpus is available offline, so every benchmark / parity input is generated from a fixed seed:
  js48k      48 944 B minified-JS-shaped text          (config 1)
  enwik      XML/wiki-shaped text, any size            (config 2: 100 000 000 B)
  mozilla    tar-like mixed binary/text, any size      (config 3: 51 220 480 B)
  mix        alternating enwik / mozilla segments      (config 4: 1 GiB)
  batch      independent 4-64 KiB payloads             (config 5: 100 000 payloads)
All generators are numpy-vectorised and return `bytes`/uint8 arrays.
"""
import numpy as np

SEED_JS, SEED_ENWIK, SEED_MOZ, SEED_MIX, SEED_BATCH = 0x5A170001, 0x5A170002, 0x5A170003, 0x5A170004, 0x5A170005


_ZIPF_CDF = {}


def _zipf_ids(rng, n, vocab, s=1.1):
    cdf = _ZIPF_CDF.get((vocab, s))
    if cdf is None:      # the table depends on (vocab, s) only: computing it once per page cost half the generator's time
        w = 1.0 / np.arange(1, vocab + 1) ** s
        cdf = np.cumsum(w)
        cdf /= cdf[-1]
        _ZIPF_CDF[(vocab, s)] = cdf
    return np.searchsorted(cdf, rng.random(n)).astype(np.int64)


def _make_vocab(rng, vocab, alphabet, minlen, maxlen):
    lens = rng.integers(minlen, maxlen + 1, size=vocab)
    # frequent words are short
    lens = np.sort(lens)
    starts = np.concatenate(([0], np.cumsum(lens)))[:-1]
    chars = alphabet[rng.integers(0, len(alphabet), size=int(lens.sum()))]
    return chars, starts, lens


def _emit_words(ids, chars, starts, lens, sep):
    """Concatenate vocabulary words ids[] each followed by the separator byte sep[i] (0 = none)."""
    L = lens[ids] + (sep != 0)
    total = int(L.sum())
    out = np.empty(total, dtype=np.uint8)
    ends = np.cumsum(L)
    begs = ends - L
    # index of the word each output byte belongs to
    widx = np.repeat(np.arange(len(ids)), L)
    k = np.arange(total) - begs[widx]
    is_sep = k >= lens[ids][widx]
    src = starts[ids][widx] + np.minimum(k, lens[ids][widx] - 1)
    out[:] = chars[src]
    out[is_sep] = sep[widx[is_sep]]
    return out


_ALPHA_LOWER = np.frombuffer(b"etaoinshrdlcumwfgypbvkjxqz", dtype=np.uint8)


def enwik(n, seed=SEED_ENWIK):
    """XML/wiki-shaped text: <page> skeletons around Zipf-distributed words with [[links]], {{templates}}, entities."""
    rng = np.random.default_rng(seed)
    chars, starts, lens = _make_vocab(rng, 50000, _ALPHA_LOWER, 2, 11)
    out = []
    have = 0
    page = 0
    while have < n:
        nwords = int(rng.integers(200, 6000))
        ids = _zipf_ids(rng, nwords, 50000)
        sep = np.full(nwords, 32, dtype=np.uint8)
        r = rng.random(nwords)
        sep[r < 0.08] = ord(",")
        sep[r < 0.045] = ord(".")
        sep[r < 0.012] = 10
        body = _emit_words(ids, chars, starts, lens, sep)
        # sprinkle markup
        marks = [b"[[", b"]]", b"{{", b"}}", b"&quot;", b"''", b"== ", b" ==\n", b"&lt;ref&gt;", b"&lt;/ref&gt;", b"|", b"*"]
        pieces = []
        cuts = np.sort(rng.integers(0, len(body), size=max(1, nwords // 25)))
        prev = 0
        for c in cuts:
            pieces.append(body[prev:c].tobytes())
            pieces.append(marks[int(rng.integers(0, len(marks)))])
            if rng.random() < 0.15:
                pieces.append(str(int(rng.integers(1000, 2021))).encode())
            prev = c
        pieces.append(body[prev:].tobytes())
        text = b"".join(pieces)
        title = _emit_words(_zipf_ids(rng, 3, 50000), chars, starts, lens, np.full(3, 32, dtype=np.uint8)).tobytes().strip().title()
        page += 1
        hdr = (b"  <page>\n    <title>" + title + b"</title>\n    <id>" + str(page * 7 + 11).encode() +
               b"</id>\n    <revision>\n      <id>" + str(15898000 + page * 13).encode() +
               b"</id>\n      <timestamp>2006-02-" + b"%02d" % (1 + page % 28) + b"T12:" + b"%02d" % (page % 60) +
               b":07Z</timestamp>\n      <contributor>\n        <username>" + title.split(b" ")[0] +
               b"</username>\n        <id>" + str(page % 9973).encode() + b"</id>\n      </contributor>\n"
               b"      <text xml:space=\"preserve\">")
        ftr = b"</text>\n    </revision>\n  </page>\n"
        blob = hdr + text + ftr
        out.append(blob)
        have += len(blob)
    return np.frombuffer(b"".join(out)[:n], dtype=np.uint8).copy()


def _opcode_markov(rng, n):
    """x86-like byte stream: opcode-biased bytes with 4-byte little-endian addresses from small pools."""
    common = np.array([0x8B, 0x89, 0xE8, 0xFF, 0x00, 0x48, 0x83, 0x0F, 0x85, 0x74, 0x24, 0x44, 0xC3, 0x55, 0x5D, 0x8D, 0xEB, 0x90, 0x01, 0x10], dtype=np.uint8)
    b = rng.integers(0, 256, size=n).astype(np.uint8)
    sel = rng.random(n)
    b[sel < 0.6] = common[rng.integers(0, len(common), size=int((sel < 0.6).sum()))]
    # address pool insertions
    pool = rng.integers(0x08040000, 0x08090000, size=64).astype("<u4")
    npts = n // 24
    at = np.sort(rng.integers(0, max(1, n - 4), size=npts))
    vals = pool[rng.integers(0, 64, size=npts)].view(np.uint8).reshape(-1, 4)
    for k in range(4):
        b[np.minimum(at + k, n - 1)] = vals[:, k]
    return b


def mozilla(n, seed=SEED_MOZ):
    """tar-like mixed binary: code, padding runs, string tables, records, text, high-entropy segments."""
    rng = np.random.default_rng(seed)
    out = []
    have = 0
    chars, starts, lens = _make_vocab(rng, 4000, np.frombuffer(b"abcdefghijklmnopqrstuvwxyz_ABCDEFGHIJ", dtype=np.uint8), 3, 14)
    while have < n:
        seg = int(np.exp(rng.uniform(np.log(4096), np.log(4 << 20))))
        seg = min(seg, n - have)
        kind = rng.random()
        if kind < 0.45:
            b = _opcode_markov(rng, seg)
        elif kind < 0.55:
            parts = []
            got = 0
            while got < seg:
                run = int(np.exp(rng.uniform(np.log(16), np.log(65536))))
                run = min(run, seg - got)
                parts.append(np.full(run, 0x00 if rng.random() < 0.7 else 0xFF, dtype=np.uint8))
                got += run
                if got < seg:
                    g = min(int(rng.integers(4, 200)), seg - got)
                    parts.append(rng.integers(0, 256, size=g).astype(np.uint8))
                    got += g
            b = np.concatenate(parts)
        elif kind < 0.70:
            nw = seg // 6 + 1
            ids = _zipf_ids(rng, nw, 4000, 1.0)
            b = _emit_words(ids, chars, starts, lens, np.zeros(nw, dtype=np.uint8) + (0 if False else 1))[:seg]
            b[b == 1] = 0
            if rng.random() < 0.4:   # UTF-16-like
                w = np.zeros(seg, dtype=np.uint8)
                w[0::2] = b[: (seg + 1) // 2]
                b = w
        elif kind < 0.85:
            nrec = seg // 16 + 1
            rec = np.zeros((nrec, 16), dtype=np.uint8)
            idx = np.arange(nrec, dtype=np.uint32) + int(rng.integers(0, 1 << 20))
            rec[:, 0:4] = idx.astype("<u4").view(np.uint8).reshape(-1, 4)
            rec[:, 4:8] = (idx * 16 + 0x1000).astype("<u4").view(np.uint8).reshape(-1, 4)
            rec[:, 8] = rng.integers(0, 4, size=nrec)
            rec[:, 12:14] = rng.integers(0, 256, size=(nrec, 2))
            b = rec.reshape(-1)[:seg]
        elif kind < 0.95:
            b = enwik(seg, seed=int(rng.integers(1, 1 << 30)))
        else:
            b = rng.integers(0, 256, size=seg).astype(np.uint8)
        out.append(b[:seg])
        have += seg
    res = np.concatenate(out)[:n]
    if len(res) < n:   # some segment kinds come out a little short of their nominal size: top up with further segments
        res = np.concatenate([res, mozilla(n - len(res), seed=seed + 7919)])
    return res.copy()


def js48k(n=48944, seed=SEED_JS):
    """Minified-JS-shaped text: identifiers, keywords, punctuation, quoted class-like strings, no whitespace."""
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ$_", dtype=np.uint8)
    nid = 400
    id_lens = np.sort(rng.integers(1, 13, size=nid))
    ids = [alpha[rng.integers(0, len(alpha), size=int(l))].tobytes() for l in id_lens]
    kws = [b"function", b"return", b"var", b"this", b"if", b"else", b"for", b"new", b"typeof", b"null", b"undefined", b"true", b"false",
           b"prototype", b"length", b"document", b"window", b"jQuery", b"call", b"apply", b"each", b"extend", b"data", b"attr", b"find",
           b"addClass", b"removeClass", b"hasClass", b"trigger", b"Event", b"target", b"options", b"element", b"parent", b"closest",
           b"case", b"break", b"while", b"in", b"instanceof"]
    punct = [b"(", b")", b"{", b"}", b";", b",", b".", b"=", b"==", b"===", b"&&", b"||", b"!", b"?", b":", b"+", b"[", b"]", b"()", b"){", b"});", b"},"]
    css = [b"\"." + b"-".join(rng.choice([b"btn", b"nav", b"modal", b"active", b"open", b"fade", b"in", b"dropdown", b"toggle", b"collapse", b"tab", b"item"],
                                         size=int(rng.integers(1, 4)))) + b"\"" for _ in range(60)]
    idw = 1.0 / np.arange(1, nid + 1) ** 1.1
    idw /= idw.sum()
    out = []
    have = 0
    while have < n:
        r = rng.random()
        if r < 0.34:
            t = ids[int(rng.choice(nid, p=idw))]
        elif r < 0.50:
            t = kws[int(rng.integers(0, len(kws)))]
        elif r < 0.93:
            t = punct[int(rng.integers(0, len(punct)))]
        elif r < 0.97:
            t = css[int(rng.integers(0, len(css)))]
        else:
            t = str(int(rng.integers(0, 1000))).encode()
        if out and out[-1][-1:].isalnum() and t[:1].isalnum():
            out.append(b" ")
            have += 1
        out.append(t)
        have += len(t)
    return np.frombuffer(b"".join(out)[:n], dtype=np.uint8).copy()


def mix(n, seed=SEED_MIX, seg_lo=8 << 20, seg_hi=64 << 20):
    """Alternating enwik / mozilla style segments (config 4)."""
    rng = np.random.default_rng(seed)
    out = []
    have = 0
    k = 0
    while have < n:
        seg = min(int(rng.integers(seg_lo, seg_hi + 1)), n - have)
        out.append(enwik(seg, seed=seed + 17 * k + 1) if k % 2 == 0 else mozilla(seg, seed=seed + 17 * k + 2))
        have += seg
        k += 1
    return np.concatenate(out)[:n].copy()


def batch(count, seed=SEED_BATCH, lo=4096, hi=65536):
    """Independent payloads: half PNG-IDAT-shaped (filter byte + small deltas), half HTTP-body-shaped text."""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(lo, hi + 1, size=count)
    text_pool = enwik(4 << 20, seed=seed + 99)
    payloads = []
    for i, sz in enumerate(sizes):
        sz = int(sz)
        if i % 2 == 0:
            width = int(rng.integers(64, 512)) * 4 + 1
            d = rng.geometric(0.35, size=sz).astype(np.int64) - 1
            sign = rng.integers(0, 2, size=sz) * 2 - 1
            b = ((d * sign) % 256).astype(np.uint8)
            b[rng.random(sz) < 0.3] = 0
            b[0::width] = rng.integers(0, 5, size=len(b[0::width]))
            payloads.append(b)
        else:
            o = int(rng.integers(0, len(text_pool) - sz))
            payloads.append(text_pool[o:o + sz].copy())
    return payloads


def batch_dictionary(n, seed=SEED_BATCH):
    """A preset dictionary for batch(count, seed): n bytes at a seeded offset of the text pool its text payloads are cut from."""
    text_pool = enwik(4 << 20, seed=seed + 99)
    o = int(np.random.default_rng(seed + 7).integers(0, len(text_pool) - n + 1))
    return text_pool[o:o + n].copy()


def lz_selftest(n, seed, alphabet, match_prob):
    """Data of the reference's self-test shape (tool/zultra.c:425-463): random literals over `alphabet` symbols mixed
    with copies of earlier data."""
    rng = np.random.default_rng(seed)
    out = bytearray()
    while len(out) < n:
        if len(out) > 10 and rng.random() < match_prob:
            ln = int(rng.integers(3, 64))
            off = int(rng.integers(1, min(len(out), 32768) + 1))
            for _ in range(ln):
                out.append(out[-off])
        else:
            out.append(int(rng.integers(0, alphabet)))
    return np.frombuffer(bytes(out[:n]), dtype=np.uint8).copy()
