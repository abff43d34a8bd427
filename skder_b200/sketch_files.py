"""skani-style per-input sketch files: `sketch -o DB` writes DB/<basename>.sketch for every input, and triangle and dist
take such a file wherever they take a FASTA (DESIGN.md section 3).  This module is the only one that writes or reads
them.

A descriptor is a small JSON object that names genomes of the database beside it; the seeds and markers stay in
DB/sketches.skb:
  format        FORMAT
  path          the input exactly as `sketch` was given it: the label its genomes take (Ref_file / Query_file)
  per_sequence  whether the database was sketched with -i (then its genomes are the file's records)
  ids           the database genome ids of that input's first occurrence: one id, or with -i its records' ids
  names         the manifest's names of those ids (Ref_name / Query_name)
  stamp         the database it belongs to: skb_db_info's digest of sketches.skb's header and tables, and the SHA-256
                of manifest.json
A descriptor whose stamp does not match the database in its directory (one left over from an earlier `sketch` into that
directory) is refused.
"""
import hashlib
import json
import os

FORMAT = "skb200-sketch-1"
SUFFIX = ".sketch"


class StaleSketch(ValueError):
    pass


def is_sketch(path):
    return path.endswith(SUFFIX)


def file_names(paths):
    """{path: descriptor file name} of every distinct path, in first-occurrence order: the first path with a given
    basename gets `<basename>.sketch`, later ones `<basename>.1.sketch`, `<basename>.2.sketch`, ... (the first such name
    no earlier path took)"""
    names, taken = {}, set()
    for p in paths:
        if p in names:
            continue
        base, k = os.path.basename(p), 0
        name = base + SUFFIX
        while name in taken:
            k += 1
            name = "%s.%d%s" % (base, k, SUFFIX)
        taken.add(name)
        names[p] = name
    return names


def _db_state(db_dir):
    """(genome count, m, stamp) of the database in db_dir as it is now"""
    from . import engine

    n, m, digest = engine.db_info(db_dir)
    with open(os.path.join(db_dir, "manifest.json"), "rb") as f:
        return n, m, "%016x:%s" % (digest, hashlib.sha256(f.read()).hexdigest())


def stamp(db_dir):
    return _db_state(db_dir)[2]


_read_dbs = {}  # db_dir -> _db_state, read once per process: a command names thousands of sketches of one database


def write_all(db_dir, inputs, paths, names, per_sequence, write):
    """One descriptor per distinct entry of `inputs` (the files as given to `sketch`, in order) for the database just
    written to db_dir, whose genome i has the manifest's paths[i] and names[i].  write(path, text) writes one file."""
    st = stamp(db_dir)
    ids = {}
    for g, p in enumerate(paths):
        ids.setdefault(p, []).append(g)
    if per_sequence:  # a file listed k times holds k copies of its records: its first occurrence owns the first copy
        reps = {}
        for p in inputs:
            reps[p] = reps.get(p, 0) + 1
        ids = {p: g[:len(g) // reps[p]] for p, g in ids.items()}
    for p, name in file_names(inputs).items():
        gi = ids.get(p, [])[:None if per_sequence else 1]
        d = {"format": FORMAT, "path": p, "per_sequence": bool(per_sequence), "ids": gi, "names": [names[g] for g in gi],
             "stamp": st}
        write(os.path.join(db_dir, name), json.dumps(d) + "\n")


class Descriptor:
    """a checked descriptor: db (its directory), path, per_sequence, ids, names, m (the database's marker compression)"""

    def __init__(self, sketch_path):
        self.file = sketch_path
        self.db = os.path.dirname(sketch_path) or "."
        try:
            with open(sketch_path) as f:
                d = json.load(f)
        except (OSError, ValueError) as e:
            raise ValueError("cannot read sketch %s: %s" % (sketch_path, e))
        if not isinstance(d, dict) or d.get("format") != FORMAT:
            raise ValueError("%s is not a %s sketch file" % (sketch_path, FORMAT))
        self.path, self.per_sequence, self.ids, self.names = d["path"], bool(d["per_sequence"]), list(d["ids"]), list(d["names"])
        if self.db not in _read_dbs:
            _read_dbs[self.db] = _db_state(self.db)
        n, self.m, st = _read_dbs[self.db]
        if d["stamp"] != st:
            raise StaleSketch("%s does not belong to the sketch database in %s (it was written for an earlier one)"
                              % (sketch_path, self.db))
        if len(self.names) != len(self.ids) or not all(isinstance(g, int) and 0 <= g < n for g in self.ids):
            raise ValueError("%s: malformed genome list" % sketch_path)
