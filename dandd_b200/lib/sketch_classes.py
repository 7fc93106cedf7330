"""Sketch objects: naming/layout of the sketch database plus the operations that fill it.

Drop-in for the reference module of the same name (reference lib/sketch_classes.py).  The class
names, constructor signatures, attributes and on-disk side effects are the reference's; the
difference is HOW a sketch gets made: where the reference builds a shell command for dashing / kmc /
kmc_tools and runs it through subprocess, these classes call the B200 SketchStore
(dandd_b200/store.py -> C ABI -> CUDA).  The command string the reference would have run is still
recorded in `.cmd` (it appears in DandD's CSV output and documents what was replaced).

    SketchFilePath            reference :31-121   (names, directories, fastahex/sketchinfo registration)
    SketchObj                 reference :124-297  (create-or-reuse, cardinality cache)
    DashSketchObj             reference :302-373  (HyperLogLog, `dashing sketch|union|card`)
    KMCSketchObj              reference :377-465  (exact, `kmc`, `kmc_tools info|complex`)
"""
import contextlib
import glob
import os

from species_specifics import SpeciesSpecifics

from dandd_b200 import ingest


def get_store():
    """The process-wide sketch store (dandd_b200.store), imported on first use: a run that is served
    entirely from the sketch database -- or ends in an argument error -- never pays for importing
    torch and starting CUDA."""
    from dandd_b200.store import get_store as _get
    return _get()


_family = None   # the exact family registered by the running hill-climb (exact_family), entered in the store on demand


@contextlib.contextmanager
def exact_family(genomes, canon: bool, sets=(), orderings=()):
    """Register the genome sets an exact hill-climb is going to count (GpuSketchStore.exact_family: `sets` are index
    lists into genomes, `orderings` index sequences whose prefixes are the sets).  Recorded here on the host: the
    store is only given the family when a count is actually computed (KMCSketchObj.build_db), so a run served
    from the sketch database never creates it.  While one family is registered another registers nothing."""
    global _family
    if _family is not None:
        yield
        return
    _family = {"args": (list(genomes), bool(canon), [list(s) for s in sets], [list(o) for o in orderings]), "open": None}
    try:
        yield
    finally:
        fam, _family = _family, None
        if fam["open"] is not None:
            fam["open"].__exit__(None, None, None)


def _store_with_family():
    """get_store(), with the registered exact family handed to it first (stores without exact_family: never)."""
    store = get_store()
    if _family is not None and _family["open"] is None and hasattr(store, "exact_family"):
        ctx = store.exact_family(*_family["args"])
        ctx.__enter__()
        _family["open"] = ctx
    return store


DASHINGLOC = "dashing"   # kept for API compatibility; only ever used inside the recorded .cmd text

_made_dirs = set()


def ensure_dir(path: str) -> None:
    """os.makedirs(exist_ok=True), once per directory and process (a progressive run asks for the
    same few hundred ngen*/k* directories tens of thousands of times)."""
    if path and path not in _made_dirs:
        os.makedirs(path, exist_ok=True)
        _made_dirs.add(path)


def nonempty_file(path: str) -> bool:
    """exists-and-not-empty with a single stat (the reference's sketch existence test, :331)."""
    try:
        return os.stat(path).st_size != 0
    except OSError:
        return False


def blake2b(fname):
    """Hex digest of the file bytes that names a FASTA (reference :12-18).  Computed by the ingest
    pool while earlier files are being sketched (dandd_b200/ingest.py); same digest."""
    return ingest.digest(fname)


def canon_command(canon: bool, tool="dashing"):
    """Flag that switches canonicalisation off for the given tool (reference :20-29)."""
    if canon:
        return ""
    return {"dashing": "--no-canon", "kmc": "-b"}.get(tool, "")


def _k_token(kval: int) -> str:
    """k as it appears in names; 0 is the '{}' placeholder of a k-sweep template (reference :43-47)."""
    return "{}" if kval == 0 else str(kval)


class SketchFilePath:
    """Where the sketch of a set of FASTAs at one k lives:  <sketchdir>/ngen<N>/k<K>/<base><ext>."""

    def __init__(self, filenames: list, kval: int, speciesinfo: SpeciesSpecifics, experiment: dict, prefix=None):
        self.ffiles = filenames
        self.files = sorted(os.path.basename(f) for f in self.ffiles)
        self.ngen = len(filenames)
        ktok = _k_token(kval)
        self.dir = os.path.join(speciesinfo.sketchdir, "ngen" + str(self.ngen), "k" + ktok)
        self.base = self._assign_base(speciesinfo=speciesinfo, kval=kval, registers=experiment["registers"],
                                      canonicalize=experiment["canonicalize"], tool=experiment["tool"],
                                      safety=experiment["safety"])
        ext = self._get_ext(experiment["tool"])
        self.relative = os.path.join("ngen" + str(self.ngen), "k" + str(kval), self.base) + ext
        self.full = os.path.join(self.dir, self.base) + ext
        if kval != 0:
            ensure_dir(self.dir)

    def __repr__(self):
        return (f"{self.__class__.__name__}[basename: {self.base}, 'fullpath inputs: {self.ffiles}', "
                f"ngen: {self.ngen}, dir: {self.dir}, fullpath: {self.full} ]")

    def _get_ext(self, tool) -> str:
        try:
            return {"dashing": ".hll", "kmc": ""}[tool]
        except KeyError:
            raise ValueError("is there another option for tool other than kmc or dashing?")

    def _hashsum(self, speciesinfo: SpeciesSpecifics):
        """blake2b of the file for one FASTA; for a set, the sum of the members' digests read as
        integers and printed with hex() -- '0x' prefix included (reference :69-78)."""
        if self.ngen == 1:
            return blake2b(self.ffiles[0])
        return hex(sum(int(speciesinfo.fastahex[name], 16) for name in self.files))

    def _assign_base(self, speciesinfo: SpeciesSpecifics, kval: int, registers: int, canonicalize: bool, tool: str,
                     safety=False) -> str:
        ktok = _k_token(kval)
        set_key = "".join(self.files)
        if set_key in speciesinfo.fastahex:
            stored = speciesinfo.fastahex[set_key]
            if safety:
                fresh = self._hashsum(speciesinfo)
                if fresh != stored:
                    raise RuntimeError(f"Checksum does not match stored value for {set_key}: {fresh}, {stored}")
        else:
            stored = speciesinfo.fastahex[set_key] = self._hashsum(speciesinfo)

        nc = "" if canonicalize else "nc"
        if self.ngen == 1:
            # dashing names single-input sketches itself; the same stem is used for kmc (reference :98-104)
            if tool == "dashing":
                sketchbase = f"{self.files[0]}.w.{ktok}.spacing.{registers}"
            else:
                sketchbase = f"{self.files[0]}_k{ktok}{nc}"
        else:
            sketchbase = f"{stored[:15]}_{registers}n{self.ngen}k{ktok}{nc}"

        info = {"sketchbase": sketchbase, "files": self.files, "ngen": self.ngen, "kval": kval, "registers": registers}
        known = speciesinfo.sketchinfo.get(sketchbase)
        if known is None:
            speciesinfo.sketchinfo[sketchbase] = info
        elif safety:
            for field, value in known.items():
                if value != info[field]:
                    raise RuntimeError(f"Duplicate keys but not duplicate values: {sketchbase}: (1) {known}, (2) {info}")
        return sketchbase


class SketchObj(object):
    """One sketch (or exact k-mer set) of one FASTA set at one k.

    Attributes (as pickled by the reference): kval, sketch (path), cmd, sfp, delta_pos, card,
    speciesinfo, experiment, _presketches.  Building an object with kval > 0 guarantees that the
    file at sfp.full exists and that speciesinfo.cardkey[sfp.full] holds its cardinality."""

    def __init__(self, kval: int, sfp: SketchFilePath, speciesinfo: SpeciesSpecifics, experiment: dict, presketches=[]):
        self.kval = kval
        self.sketch = None
        self.cmd = None
        self.sfp = sfp
        self.delta_pos = 0
        self.card = 0
        self.speciesinfo = speciesinfo
        experiment["baseset"].add(sfp.base)
        self.experiment = experiment
        self._presketches = presketches
        if self.kval > 0:
            self.create_sketch()
            self.card = self.check_cardinality()
            self.delta_pos = self.card / self.kval

    def __lt__(self, other):
        return self.delta_pos < other.delta_pos

    def __gt__(self, other):
        return self.delta_pos > other.delta_pos

    def __repr__(self):
        return (f"['sketch loc: {self.sketch}', k: {self.kval}, pos delta: {self.delta_pos}, "
                f"cardinality: {self.card}, command: {self.cmd}  ]")

    # -- supplied by the tool-specific subclasses ----------------------------------------------------
    def sketch_check(self, path=None) -> bool:
        raise NotImplementedError("Subclass needs to define this.")

    def _leaf_command(self, tmpdir) -> str:
        raise NotImplementedError("Subclass needs to define this.")

    def _union_command(self) -> str:
        raise NotImplementedError("Subclass needs to define this.")

    def card_command(self, sketch_paths=[]):
        raise NotImplementedError("Subclass must define this.")

    def parse_card(self, proc):
        raise NotImplementedError("Subclass must define this.")

    def remove_sketch(self):
        raise NotImplementedError("Subclass must define this.")

    def _run_leaf(self) -> None:
        """Make the leaf sketch exist (the GPU stand-in for running _leaf_command())."""
        raise NotImplementedError("Subclass needs to define this.")

    def _run_union(self) -> None:
        """Make the union sketch exist (the GPU stand-in for running _union_command())."""
        raise NotImplementedError("Subclass needs to define this.")

    def _run_card(self) -> None:
        """Store this sketch's cardinality in cardkey (stand-in for card_command + parse_card)."""
        raise NotImplementedError("Subclass needs to define this.")

    # -- create-or-reuse (reference :177-247) -----------------------------------------------------------
    def _say(self, flag: str, text: str) -> None:
        if self.experiment.get(flag):
            print(text)

    def _leaf_sketch(self, just_do_it=False):
        cmd = self._leaf_command(tmpdir="")
        self._say("debug", cmd)
        if just_do_it:
            self._say("verbose", "Due to issues with leaf sketch/db file, we will Just Do It. (It=Sketch or Build Again)")
            self._run_leaf()
        elif not self.sketch_check():
            trusted = self.experiment["lowmem"] and self.check_cardinality() > 0
            if not trusted:
                self._say("verbose", "Running Leaf Command: " + cmd)
                self._run_leaf()
        self.cmd = cmd   # recorded whether or not anything had to run

    def _union_sketch(self, just_do_it=False):
        cmd = self._union_command()
        if just_do_it:
            self._run_union()
            self.cmd = cmd
        elif not self.sketch_check():
            trusted = self.experiment["lowmem"] and self.check_cardinality() > 0
            if not trusted:
                self._say("verbose", "Running Union Command: " + cmd)
                self._run_union()
            self.cmd = cmd   # only when the union was missing (reference :223-232: cached => None)
        self._say("debug", self.cmd)

    def create_sketch(self, just_do_it=False):
        if self.sfp.ngen == 1:
            self._leaf_sketch(just_do_it=just_do_it)
        elif self.sfp.ngen > 1:
            self._union_sketch(just_do_it=just_do_it)
        else:
            raise RuntimeError("For some reason you are trying to sketch an empty list of files. Don't do that.")
        self.sketch = self.sfp.full
        return self.sketch

    # -- cardinality cache (reference :254-297) ---------------------------------------------------------
    def individual_card(self, cmd=None) -> None:
        """Compute and store the cardinality of this sketch; if that fails (unreadable sketch
        file) rebuild the sketch once and try again (reference :267-278)."""
        if self.kval == 0:
            return
        self._say("debug", cmd or self.card_command())
        try:
            self._run_card()
        except (OSError, ValueError, RuntimeError):
            print(f"Recreating sketch {self.sfp.full}")
            self.create_sketch(just_do_it=True)
            self._run_card()

    def check_cardinality(self) -> float:
        key = self.sfp.full
        cardkey = self.speciesinfo.cardkey
        if key not in cardkey and self.experiment["lowmem"]:
            return 0
        stored = cardkey.get(key)
        if stored is None or float(stored) == 0:
            if not self.sketch_check():
                return 0
            self.individual_card()
        self.card = float(cardkey[key])
        self.delta_pos = self.card / int(self.kval)
        return float(self.card)


class DashSketchObj(SketchObj):
    """HyperLogLog sketch, bit-identical to `dashing sketch -k K -S registers` (SURVEY.md App. A)."""

    def __init__(self, kval, sfp, speciesinfo, experiment, presketches=[]):
        super().__init__(kval=kval, sfp=sfp, speciesinfo=speciesinfo, experiment=experiment, presketches=presketches)

    # command text (recorded, never executed)
    def card_command(self, sketch_paths=[]) -> str:
        if len(sketch_paths) == 0:
            if self.kval == 0:
                return
            sketch_paths = [self.sketch]
        return " ".join([DASHINGLOC, "card", "--presketched"] + sketch_paths)

    def _leaf_command(self, tmpdir) -> str:
        parts = [DASHINGLOC, "sketch", canon_command(self.experiment["canonicalize"], "dashing"),
                 "-k" + _k_token(self.kval), "-S", str(self.experiment["registers"]), "--prefix", str(self.sfp.dir),
                 self.sfp.ffiles[0]]
        return " ".join(parts)

    def _union_command(self) -> str:
        return " ".join([DASHINGLOC, "union", "-z -o", str(self.sfp.full)] + self._presketches)

    def parse_card(self, proc):
        """Accepts the text `dashing card` prints (reference :318-321), for callers that still have it."""
        lines = proc.stdout.splitlines()
        for line in lines[1:]:
            path, _, size = line.partition("\t")
            self.speciesinfo.cardkey[path] = float(size)

    # GPU-backed operations
    def _run_leaf(self) -> None:
        cards = get_store().leaf_sketches(self.sfp.ffiles[0], [self.kval], int(self.experiment["registers"]),
                                          bool(self.experiment["canonicalize"]), {self.kval: self.sfp.full})
        self.speciesinfo.cardkey[self.sfp.full] = cards[self.kval]

    def _run_union(self) -> None:
        cards = get_store().union_sketches({self.kval: list(self._presketches)}, int(self.experiment["registers"]),
                                           {self.kval: self.sfp.full})
        self.speciesinfo.cardkey[self.sfp.full] = cards[self.kval]

    def _run_card(self) -> None:
        self.speciesinfo.cardkey[self.sfp.full] = get_store().card_of_file(self.sfp.full)

    def sketch_check(self, path=None) -> bool:
        path = path or self.sfp.full
        return nonempty_file(path)

    def remove_sketch(self, delete_me: str = None):
        pattern = delete_me or self.sfp.full
        if self.kval == 0:
            pattern = self.sfp.full.replace("{}", "*")
        for hit in glob.glob(pattern):
            try:
                os.remove(hit)
            except FileNotFoundError:
                pass
            get_store().forget(hit)


class KMCSketchObj(SketchObj):
    """Exact mode: the number of distinct (canonical) k-mers, KMC semantics (SURVEY.md App. B).
    The "database" written at sfp.full + .kmc_pre/.kmc_suf is a small descriptor (k, flags, member
    FASTAs, count), not a KMC database: DandD only ever asks for its existence and its size."""

    MAGIC = b"DANDD-B200 exact k-mer set v1\n"

    def __init__(self, kval, sfp, speciesinfo, experiment, presketches=[]):
        super().__init__(kval=kval, sfp=sfp, speciesinfo=speciesinfo, experiment=experiment, presketches=presketches)

    # command text (recorded, never executed)
    def _tflag(self) -> str:
        n = self.experiment["nthreads"]
        return " -t" + str(n) if n > 0 else ""

    def card_command(self, sketch_paths: list = []) -> str:
        if len(sketch_paths) == 0:
            if self.kval == 0:
                return
            sketch_paths = [self.sketch]
        return ("for db in " + " ".join(sketch_paths) + "; do value=$(kmc_tools -hp info $db | grep 'total k-mers' | "
                "sed 's/ //g' | sed 's/totalk-mers://g'); echo $db,$value; done")

    def _leaf_command(self, tmpdir) -> str:
        ktok = _k_token(self.kval)
        parts = ["kmc -hp" + self._tflag(), " -ci1 -cs2", "-k" + ktok, canon_command(self.experiment["canonicalize"], "kmc"),
                 "-fm", self.sfp.ffiles[0], self.sfp.full, os.path.join(tmpdir, "k" + ktok)]
        return " ".join(parts)

    def _union_command(self) -> str:
        lines = ["INPUT: "] + [f"input{i + 1} = {db} -ci1   " for i, db in enumerate(self._presketches)]
        expr = " + ".join(f"input{i + 1}" for i in range(len(self._presketches)))
        spec = "\n".join(lines) + f"\nOUTPUT:\n{self.sfp.full} = {expr}"
        return " ".join([f'echo -e "{spec}"', "|", "kmc_tools", "-hp ", self._tflag(), "complex", "/dev/stdin"])

    def parse_card(self, proc):
        for line in proc.stdout.splitlines():
            path, value = line.strip().split(",")
            self.speciesinfo.cardkey[path] = float(value)

    # GPU-backed operations
    @classmethod
    def build_db(cls, full: str, kval: int, canon: bool, fastas, cardkey) -> int:
        """Count the distinct k-mers of the FASTA set on the GPU, write the descriptor pair at
        `full` + .kmc_pre/.kmc_suf and cache the count -- `kmc` (one FASTA) or `kmc_tools complex`
        (several) followed by `kmc_tools info`, in one step."""
        count = _store_with_family().exact_count(list(fastas), kval, canon)
        cls.write_db(full, kval, canon, fastas, count, cardkey)
        return count

    @classmethod
    def write_db(cls, full: str, kval: int, canon: bool, fastas, count: int, cardkey) -> None:
        """Write the descriptor pair of a set whose count is known at `full` + .kmc_pre/.kmc_suf and cache
        the count (build_db, and the pairs a batched all-pairs job has already counted).  cardkey=None: the
        count is left for the object that later finds the descriptor to read back (_run_card)."""
        ensure_dir(os.path.dirname(full))
        body = (cls.MAGIC + f"k={kval}\ncanonical={int(canon)}\ntotal k-mers={count}\n".encode()
                + "".join(f"input={f}\n" for f in fastas).encode())
        for ext in (".kmc_pre", ".kmc_suf"):
            with open(full + ext, "wb") as fh:
                fh.write(body)
        if cardkey is not None:
            cardkey[full] = float(count)

    def _run_leaf(self) -> None:
        self.build_db(self.sfp.full, self.kval, bool(self.experiment["canonicalize"]), self.sfp.ffiles,
                      self.speciesinfo.cardkey)

    _run_union = _run_leaf   # a union database is the set of all member FASTAs' k-mers

    def _run_card(self) -> None:
        """`kmc_tools info`: read the count back from the descriptor, else recount."""
        try:
            with open(self.sfp.full + ".kmc_pre", "rb") as fh:
                for line in fh.read().split(b"\n"):
                    if line.startswith(b"total k-mers="):
                        self.speciesinfo.cardkey[self.sfp.full] = float(line.split(b"=")[1])
                        return
        except OSError:
            pass
        self._run_leaf()

    def sketch_check(self, path=None) -> bool:
        """Both database files exist and are non-empty.  (The reference additionally calls
        check_cardinality() here, which calls sketch_check() again: a RecursionError as shipped,
        SURVEY.md App. B; the intended existence test is what is implemented.)"""
        path = path or self.sfp.full
        return all(nonempty_file(path + ext) for ext in (".kmc_pre", ".kmc_suf"))

    def remove_sketch(self, delete_me: str = None):
        pattern = delete_me or self.sfp.full
        if self.kval == 0:
            pattern = self.sfp.full.replace("{}", "*")
        for hit in glob.glob(pattern + ".kmc_*"):
            try:
                os.remove(hit)
            except FileNotFoundError:
                pass
