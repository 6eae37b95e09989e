"""TEST INFRASTRUCTURE: the reference's release artefacts and a sample of its proof files, stored under tests/golden
(tests/golden/make_reference_proofs.py says what was kept).  REL holds release-v0.13.1's files as shipped; proof_files_dir() writes the
proof files, in the reference's own JSON layout, to a temporary directory that lives as long as the test process."""
import atexit
import json
import os
import shutil
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REL = os.path.join(HERE, "golden", "release-v0.13.1")
GOLD = json.load(open(os.path.join(HERE, "golden", "reference_proofs.json")))
_DIR = []


def proof_files_dir() -> str:
    if not _DIR:
        d = tempfile.mkdtemp(prefix="reference_test_data_")
        atexit.register(shutil.rmtree, d, True)
        for name, content in GOLD["files"].items():
            content = json.loads(json.dumps(content))
            for e in content.get("chunk_proofs", []) + ([content] if "protocol" in content else []):
                e["protocol"] = GOLD["shared"][e["protocol"]]
            os.makedirs(os.path.dirname(os.path.join(d, name)), exist_ok=True)
            with open(os.path.join(d, name), "w") as f:
                json.dump(content, f)
        _DIR.append(d)
    return _DIR[0]
