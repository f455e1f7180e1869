"""Regenerates tests/golden/handmade_set.json: the 43 `$set` lines of the reference's data/sample-handmade-data.txt as
[item, property, value], parsed as examples/import_handmade.py:47-57 does (values split on ':', defaultRank a float).
Run where the reference tree is mounted; the other golden files are not touched."""
import json
import os

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    rows = []
    for line in open(f"{REF}/data/sample-handmade-data.txt"):
        data = line.rstrip("\r\n").split(",")
        if len(data) == 3 and data[1] == "$set":
            props = data[2].split(":")
            name = props.pop(0)
            rows.append([data[0], name, float(props[0]) if name == "defaultRank" else props])
    json.dump({"source": "data/sample-handmade-data.txt ($set lines)", "set": rows}, open(f"{HERE}/handmade_set.json", "w"), indent=1)


if __name__ == "__main__":
    main()
