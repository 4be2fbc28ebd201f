"""Shared host-side helpers for the tests (pure Python, no oracle, no GPU)."""


def rlp_uint(i):
    """RLP of an unsigned integer (the key of an index trie, src/blockchain/blockchain.zig:214-232)."""
    if i == 0:
        return b"\x80"
    b = i.to_bytes((i.bit_length() + 7) // 8, "big")
    return b if len(b) == 1 and b[0] < 0x80 else bytes([0x80 + len(b)]) + b


def index_trie_items(values):
    """(key, value) list of an index trie, sorted the way mptize wants it."""
    return sorted(((rlp_uint(i), v) for i, v in enumerate(values)), key=lambda kv: kv[0])


# ---- a third, independent statement of the proof walk (small cases only) ----
def _rlp_item(b, pos, end):
    """strict decode; returns (is_list, payload_start, payload_end, item_end) or None"""
    if pos >= end:
        return None
    x = b[pos]
    if x < 0x80:
        return (False, pos, pos + 1, pos + 1)
    is_list = x >= 0xc0
    base_s, base_l = (0xc0, 0xf7) if is_list else (0x80, 0xb7)
    if x <= base_l:
        n = x - base_s
        if pos + 1 + n > end:
            return None
        if not is_list and n == 1 and b[pos + 1] < 0x80:
            return None
        return (is_list, pos + 1, pos + 1 + n, pos + 1 + n)
    ll = x - base_l
    if ll > 4 or pos + 1 + ll > end or b[pos + 1] == 0:
        return None
    n = int.from_bytes(b[pos + 1:pos + 1 + ll], "big")
    if n <= 55 or pos + 1 + ll + n > end:
        return None
    return (is_list, pos + 1 + ll, pos + 1 + ll + n, pos + 1 + ll + n)


EMPTY_ROOT = bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")


def py_verify(keccak, nodes, key32, root):
    """-> (status, value bytes or None); status 0 reject / 1 present / 2 absent.  See oracle/verify.c R1-R4."""
    if not nodes:
        return (2, None) if root == EMPTY_ROOT else (0, None)
    nib = [n for byte in key32 for n in (byte >> 4, byte & 15)]
    pos, i, expect = 0, 0, root
    cur, embedded = None, False
    while True:
        if not embedded:
            if i == len(nodes):
                return (0, None)
            cur = nodes[i]
            if keccak(cur) != expect:
                return (0, None)
            i += 1
        top = _rlp_item(cur, 0, len(cur))
        if top is None or not top[0] or top[3] != len(cur):
            return (0, None)
        items, p = [], top[1]
        while p < top[2]:
            it = _rlp_item(cur, p, top[2])
            if it is None or len(items) == 17:
                return (0, None)
            items.append((it, p))
            p = it[3]
        if len(items) not in (2, 17):
            return (0, None)
        last = i == len(nodes)
        if len(items) == 17:
            if pos == 64:
                it = items[16][0]
                if it[0] or not last:
                    return (0, None)
                return (2, None) if it[1] == it[2] else (1, cur[it[1]:it[2]])
            child = items[nib[pos]]
            pos += 1
        else:
            it = items[0][0]
            if it[0] or it[1] == it[2]:
                return (0, None)
            hp = cur[it[1]:it[2]]
            flag = hp[0] >> 4
            if flag > 3 or (not flag & 1 and hp[0] & 15):
                return (0, None)
            path = ([hp[0] & 15] if flag & 1 else []) + [n for byte in hp[1:] for n in (byte >> 4, byte & 15)]
            if len(path) > 64:
                return (0, None)
            match = nib[pos:pos + len(path)] == path
            if flag & 2:
                v = items[1][0]
                if v[0] or not last:
                    return (0, None)
                if match and pos + len(path) == 64:
                    return (1, cur[v[1]:v[2]])
                return (2, None)
            if not path:
                return (0, None)
            if not match:
                return (2, None) if last else (0, None)
            pos += len(path)
            child = items[1]
        it, start = child
        if it[0]:
            if it[3] - start >= 32:
                return (0, None)
            cur, embedded = cur[start:it[3]], True
            continue
        embedded = False
        n = it[2] - it[1]
        if n == 0:
            if len(items) == 2:
                return (0, None)
            return (2, None) if last else (0, None)
        if n != 32:
            return (0, None)
        expect = cur[it[1]:it[2]]


# ---- plain RLP encode (host-side test data preparation) ----
def rlp_str(b):
    if len(b) == 1 and b[0] < 0x80:
        return bytes(b)
    if len(b) <= 55:
        return bytes([0x80 + len(b)]) + bytes(b)
    ll = (len(b).bit_length() + 7) // 8
    return bytes([0xb7 + ll]) + len(b).to_bytes(ll, "big") + bytes(b)


def rlp_list(encoded_items):
    body = b"".join(encoded_items)
    if len(body) <= 55:
        return bytes([0xc0 + len(body)]) + body
    ll = (len(body).bit_length() + 7) // 8
    return bytes([0xf7 + ll]) + len(body).to_bytes(ll, "big") + body


def rlp_int_be(b):
    return rlp_str(bytes(b).lstrip(b"\x00"))


def secure_account_items(keccak, mptize, accounts):
    """(keccak(addr), rlp(account)) sorted -- the state trie's key/values
    (evmone/test/state/mpt_hash.cpp:15-36)."""
    items = []
    for a in accounts:
        st = sorted((keccak(bytes.fromhex(k)), rlp_int_be(bytes.fromhex(v)))
                    for k, v in a["storage"].items() if int(v, 16) != 0)
        sroot = mptize(st)
        body = [rlp_int_be(a["nonce"].to_bytes(8, "big")), rlp_int_be(bytes.fromhex(a["balance"])), rlp_str(sroot),
                rlp_str(keccak(bytes.fromhex(a["code"])))]
        items.append((keccak(bytes.fromhex(a["address"])), rlp_list(body)))
    return sorted(items)


# ---- an independent statement of mptize (src/mpt/mpt.zig:38-119, 132-314) in plain Python: second opinion for the C oracle ----
def _hp(nibbles, leaf):
    """hex-prefix (mpt.zig:285-314): flag nibble 0/1 extension even/odd, 2/3 leaf even/odd"""
    flag = 2 if leaf else 0
    if len(nibbles) % 2:
        nibbles = [flag + 1] + list(nibbles)
    else:
        nibbles = [flag, 0] + list(nibbles)
    return bytes((nibbles[i] << 4) | nibbles[i + 1] for i in range(0, len(nibbles), 2))


def _py_node(keccak, items, level):
    """items: sorted [(nibble list, value)] sharing their first `level` nibbles -> the node's RLP (b"" = empty)"""
    if not items:
        return b""
    if len(items) == 1:
        return rlp_list([rlp_str(_hp(items[0][0][level:], True)), rlp_str(items[0][1])])
    first, last = items[0][0], items[-1][0]
    common = level
    while common < len(first) and common < len(last) and first[common] == last[common]:
        common += 1
    common = min(common, len(first))  # a key that ends inside the shared run ends the extension there
    if common > level:
        child = _py_node(keccak, items, common)
        return rlp_list([rlp_str(_hp(first[level:common], False)), child if len(child) < 32 else rlp_str(keccak(child))])
    value = b""
    if len(first) == level:
        value, items = items[0][1], items[1:]
    slots = []
    for v in range(16):
        child = _py_node(keccak, [it for it in items if it[0][level] == v], level + 1)
        slots.append(rlp_str(b"") if not child else (child if len(child) < 32 else rlp_str(keccak(child))))
    return rlp_list(slots + [rlp_str(value)])


def py_mptize(keccak, kv):
    """kv: sorted [(key bytes, value bytes)] -> root (the root node is always hashed, mpt.zig:42; empty list -> keccak(0x80))"""
    items = [([n for b in k for n in (b >> 4, b & 15)], v) for k, v in kv]
    node = _py_node(keccak, items, 0)
    return keccak(node if node else b"\x80")


# ---- inputs whose answers were computed by the reference's own compiled code (tests/golden/compiled_reference_kat.json,
# written by tests/golden/make_compiled_reference_kat.py): changing them invalidates the stored answers
def compiled_reference_keccak_messages():
    """random messages of lengths 0..299 and around the 136-byte rate boundaries, up to 1200 bytes"""
    import numpy as np
    rng = np.random.default_rng(1)
    return [rng.integers(0, 256, n, dtype=np.uint8).tobytes()
            for n in list(range(0, 300)) + [407, 408, 409, 543, 544, 545, 1087, 1088, 1089, 1200]]


def compiled_reference_secure_tries():
    """random secure tries: sorted 32-byte keys, 33..119-byte values, 1..1000 entries -> [[(key, value)]]"""
    import numpy as np
    rng = np.random.default_rng(7)
    tries = []
    for n in (1, 2, 3, 17, 100, 1000):
        keys = sorted(rng.integers(0, 256, 32, dtype=np.uint8).tobytes() for _ in range(n))
        vals = [rng.integers(0, 256, int(rng.integers(33, 120)), dtype=np.uint8).tobytes() for _ in range(n)]
        tries.append(list(zip(keys, vals)))
    return tries


def inputs_sha256(chunks):
    """sha256 over length-prefixed byte strings: pins the inputs that stored answers belong to"""
    import hashlib
    h = hashlib.sha256()
    for c in chunks:
        h.update(len(c).to_bytes(8, "little") + c)
    return h.hexdigest()


# ---- a stand-in for phant_b200.gpu.Context that computes with the CPU oracle: lets the HOST logic above the C ABI
# (flattening, decoding, ownership, error mapping) run in the CPU test suite; the -m gpu tests run the same host code on the device
class OracleBackedCtx:
    def __init__(self, o):
        self.o = o

    def keccak256_batch(self, data, off, n, out):
        import numpy as np
        for i in range(n):
            out[i] = np.frombuffer(self.o.keccak256(data[int(off[i]):int(off[i + 1])].tobytes()), np.uint8)

    def mpt_roots(self, keys, key_off, vals, val_off, seg_off, n_tries):
        out = []
        for t in range(n_tries):
            kv = [(keys[int(key_off[i]):int(key_off[i + 1])].tobytes(), vals[int(val_off[i]):int(val_off[i + 1])].tobytes())
                  for i in range(int(seg_off[t]), int(seg_off[t + 1]))]
            out.append(self.o.mptize(kv))
        return out

    def verify_witness(self, n_nodes, nodes, node_off, n_keys, keys32, roots32, n_roots, bitmap, status, val_off, val_len):
        st = self.o.verify_bag(nodes, node_off, keys32, roots32, threads=1)[0]
        status[:] = st

    def ecrecover_batch(self, hashes32, sigs65, n, pubkeys65, addresses20, ok):
        import numpy as np
        for i in range(n):
            pub = self.o.ecrecover(hashes32[32 * i:32 * i + 32].tobytes(), sigs65[65 * i:65 * i + 65].tobytes())
            ok[i] = 1 if pub else 0
            if pubkeys65 is not None:
                pubkeys65[i] = np.frombuffer(pub or bytes(65), np.uint8)
            if addresses20 is not None:
                addresses20[i] = np.frombuffer(self.o.keccak256(pub[1:])[12:] if pub else bytes(20), np.uint8)
