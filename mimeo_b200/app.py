"""`mimeo <x|self|map|filter>` dispatcher (host mirror of src/mimeo/app.py:21-63). The tandem-repeat mask (GPU, DESIGN §2
T1-T4) filters alignments in `mimeo map --maxtandem` and whole FASTA records in `mimeo filter`."""
import sys
from importlib import import_module

COMMANDS = {'x': 'mimeo_b200.run_interspecies', 'self': 'mimeo_b200.run_self', 'map': 'mimeo_b200.run_map',
            'filter': 'mimeo_b200.run_filter'}


def print_usage():
    print('\nUsage: mimeo <command> [options]\n\nCommands:\n  x       Run cross-species comparison\n'
          '  self    Run self-alignment analysis\n  map     Run genomic mapping\n'
          '  filter  Remove tandem-repeat-rich sequences from a FASTA library\n\nFor command-specific help:\n  mimeo <command> --help\n')


def main():
    if len(sys.argv) < 2:
        print_usage()
        sys.exit(1)
    sub = sys.argv[1]
    if sub not in COMMANDS:
        print(f"Error: Unknown command '{sub}'")
        print_usage()
        sys.exit(1)
    sys.argv = [sys.argv[0]] + sys.argv[2:]
    try:
        import_module(COMMANDS[sub]).main()
    except ImportError as e:
        print(f'Error importing module {COMMANDS[sub]}: {e}')
        sys.exit(1)
    except Exception as e:
        print(f"Error running command '{sub}': {e}")
        sys.exit(1)


if __name__ == '__main__':
    main()
