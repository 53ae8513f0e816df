"""`python mr_svm.py --tables 2 4 [-v]` -- same entry point as the reference's mr_svm.py:118-165."""
import sys

from mr_gan_b200.mr_svm import main, mr_svm  # noqa: F401

if __name__ == '__main__':
    sys.exit(main())
